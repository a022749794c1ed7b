"""Micro-benchmark of individual C-ABI kernels at the bench workload's shapes (CUDA-event timed).

    python tools/kbench.py [--iters 5] [--only substr]

Prints ms / achieved GB/s (algorithmic bytes) / TFLOP/s per configuration; used to pick the next
optimisation target and as the command profiled with ncu for profiles/."""
import argparse
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import b200path  # noqa: F401,E402
import b200_native as nat  # noqa: E402

DEV = "cuda"


def conv_case(name, B, H, W, cin, cout, taps, res_mode=0, act=1, gap=False, n_split=None, up2=False, dot=False,
              store=True, drop=False):
    x = (torch.randn(B, H, W, cin, device=DEV) * 0.5).bfloat16()
    w = (torch.randn(cout, taps * cin, device=DEV) / math.sqrt(taps * cin)).bfloat16()
    scale = torch.rand(cout, device=DEV) + 0.5
    bias = torch.randn(cout, device=DEV) * 0.1
    n1 = cout if n_split is None else n_split
    res = (torch.randn(B, H, W, n1, device=DEV) * 0.5).bfloat16() if res_mode else None
    gapb = torch.zeros(B, cout, device=DEV) if gap else None
    out = torch.empty(B, H * (2 if up2 else 1), W * (2 if up2 else 1), n1, device=DEV, dtype=torch.bfloat16) if store else None
    out2 = torch.empty(B, H, W, cout - n1, device=DEV, dtype=torch.bfloat16) if n_split else None
    dw = torch.randn(9, cout, device=DEV) if dot else None
    dout = torch.empty(B, H, W, 9, device=DEV) if dot else None

    def run():
        nat.conv_gemm(x, w, taps=taps, scale=scale, bias=bias, res=res, res_mode=res_mode, act=act, out=out, up2=up2,
                      gap=gapb, n_split=n_split, act2=1, out2=out2, dot_w=dw, dot_out=dout, store=store,
                      dropout=(0.1, 7, 1) if drop else None)

    px = B * H * W
    byts = px * cin * 2 + (px * n1 * 2 * (4 if up2 else 1) if store else 0) + (px * (cout - n1) * 2 if n_split else 0) \
        + (px * n1 * 2 if res_mode else 0) + (px * 36 if dot else 0) + cout * taps * cin * 2
    flops = 2.0 * px * cout * taps * cin
    return name, run, byts, flops


def linear_mc_case(name, M, K, N):
    """Transformer proj / fc2 under MC dropout: fp32 residual stream, out = res + drop(x w^T * scale + bias)."""
    x = (torch.randn(M, K, device=DEV) * 0.5).bfloat16()
    w = (torch.randn(N, K, device=DEV) / math.sqrt(K)).bfloat16()
    scale = torch.rand(N, device=DEV) + 0.5
    bias = torch.randn(N, device=DEV) * 0.1
    res = torch.randn(M, N, device=DEV)
    out = torch.empty(M, N, device=DEV)

    def run():
        nat.linear_f32(x, w, scale=scale, bias=bias, res=res, res_mode=2, out=out, dropout=(0.1, 7))

    return name, run, M * K * 2 + M * N * 8 + N * K * 2, 2.0 * M * N * K


def vit_bench(batch, iters):
    """ViT-B/16 features_only backbone (foundation_model.B200ViTBackbone), DCE-shaped input (6 x 224 x 224)."""
    import foundation_model as fm

    bb = fm.B200ViTBackbone(in_chans=6).to(DEV).eval()
    x = torch.rand(batch, 6, 224, 224, device=DEV)
    for _ in range(2):
        bb(x)
    torch.cuda.synchronize()
    nat.start_profile()
    bb(x)
    prof = nat.stop_profile()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        bb(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    gf_case = 35.36  # SURVEY.md row a13: 2*MAC of the matmuls, per case, C=6
    print(f"ViT-B/16 backbone, batch {batch}: {ms:.2f} ms/forward, {batch / ms * 1e3:.0f} cases/s, "
          f"{batch * gf_case / ms:.0f} TFLOP/s algorithmic")
    tot = sum(sum(t) for t in prof.values())
    for (name, key), t in sorted(prof.items(), key=lambda kv: -sum(kv[1]))[:12]:
        print(f"   {sum(t):8.3f} ms {100 * sum(t) / tot:5.1f}%  x{len(t):3d}  {name} {key}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vit", type=int, default=0, help="benchmark the ViT-B/16 backbone at this batch size instead")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--only", default="")
    ap.add_argument("--batch", type=int, default=1024)
    a = ap.parse_args()
    if a.vit:
        vit_bench(a.vit, a.iters)
        return
    B = a.batch
    cases = [
        conv_case("3x3 256->256 gelu", B, 32, 32, 256, 256, 9),
        conv_case("3x3 256->256 gelu + tapdot, no store", B, 32, 32, 256, 256, 9, dot=True, store=False),
        conv_case("3x3 128->128 gelu", B, 32, 32, 128, 128, 9),
        conv_case("3x3 128->128 gelu + tapdot, no store", B, 32, 32, 128, 128, 9, dot=True, store=False),
        conv_case("3x3 64->64 gelu", B, 32, 32, 64, 64, 9),
        conv_case("1x1 256->512 +res gelu gap", B, 32, 32, 256, 512, 1, res_mode=1, gap=True),
        conv_case("1x1 256->512 +res gelu", B, 32, 32, 256, 512, 1, res_mode=1),
        conv_case("1x1 256->512 gelu", B, 32, 32, 256, 512, 1),
        conv_case("1x1 256->512 linear", B, 32, 32, 256, 512, 1, act=0),
        conv_case("1x1 256->512 linear gap", B, 32, 32, 256, 512, 1, act=0, gap=True),
        conv_case("1x1 256->768 split 512|256", B, 32, 32, 256, 768, 1, act=0, n_split=512),
        conv_case("1x1 128->256 +res gelu gap", B, 32, 32, 128, 256, 1, res_mode=1, gap=True),
        conv_case("1x1 128->256 gelu +res(after)", B, 32, 32, 128, 256, 1, res_mode=2),
        conv_case("1x1 128->384 split 256|128", B, 32, 32, 128, 384, 1, act=0, n_split=256),
        conv_case("1x1 64->128 +res gelu gap", B, 32, 32, 64, 128, 1, res_mode=1, gap=True),
        conv_case("1x1 512->128 gap (proj_in)", B, 32, 32, 512, 128, 1, act=0, gap=True),
        conv_case("1x1 256->64 bias (mask pre)", B, 32, 32, 256, 64, 1, act=0),
        conv_case("1x1 128->64 gelu (proj)", B, 32, 32, 128, 64, 1),
        conv_case("1x1 64->64 gelu up2 (proj out)", B, 32, 32, 64, 64, 1, up2=True),
        conv_case("1x1 64->64 gelu", B, 32, 32, 64, 64, 1),
        conv_case("1x1 128->128 gelu mc-dropout", B, 32, 32, 128, 128, 1, drop=True),
        conv_case("1x1 128->64 gelu mc-dropout", B, 32, 32, 128, 64, 1, drop=True),
        linear_mc_case("linear 2048->512 fp32 res mc-dropout (fc2)", B * 256, 2048, 512),
        linear_mc_case("linear 512->128 fp32 res mc-dropout", B * 256, 512, 128),
    ]
    import numpy as np
    import dataset as b_dataset
    import preprocess_helpers as b_pre
    dwi = torch.rand(B, 16, 64, 64, device=DEV) * 1000 + 1
    dce = torch.rand(B, 6, 64, 64, device=DEV)
    pm = torch.empty(B * 16, device=DEV)
    norm = b_dataset.DWINormalize()
    nyul = b_pre.NyulStandardizer()
    nyul.fit(list(dce[:16].cpu()), num_channels=6)
    cases.insert(0, ("DWI normalise 16x64x64 (+plane means)", lambda: norm.batch(dwi, plane_mean=pm), B * 31 * 16384, 0.0))
    cases.insert(1, ("DCE Nyul 6x64x64", lambda: nyul.transform_batch(dce), B * 12 * 16384, 0.0))
    print(f"{'case':42s} {'ms':>8s} {'GB/s':>8s} {'TFLOP/s':>8s}")
    for name, run, byts, flops in cases:
        if a.only and a.only not in name:
            continue
        for _ in range(2):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.iters):
            run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.iters
        print(f"{name:42s} {ms:8.3f} {byts / ms / 1e6:8.0f} {flops / ms / 1e9:8.0f}")


if __name__ == "__main__":
    main()
