"""Stand-alone timing of b200_attention (CUDA events, L2-cold by rotating buffers).

    python tools/attn_bench.py [B N heads dh] [--p P]   one shape; P > 0 times b200_attention_mc (attention dropout)
    python tools/attn_bench.py --mc                      MC-dropout costs: p = 0 and p = 0.1 alternated in one process
                                                         at the hybrid stage (B = 1024, 256 tokens, 4 x 128) and the
                                                         ViT-B/16 shape (B = 256, 197 tokens, 12 x 64), and the proj /
                                                         fc2 launches of linear_f32 (b200_linear vs b200_linear_mc)
"""
import argparse
import subprocess
import sys

import torch

sys.path.insert(0, ".")
import b200path  # noqa: F401
import b200_native as nat


def _time(fn, nbuf, reps):
    for i in range(nbuf):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i % nbuf)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def attention_case(B, N, heads, dh, nbuf=4):
    C = heads * dh
    qkv = [(torch.randn(B * N, 3 * C, device="cuda") * 0.9).bfloat16() for _ in range(nbuf)]
    out = [torch.empty(B * N, C, device="cuda", dtype=torch.bfloat16) for _ in range(nbuf)]
    return lambda p, reps=20: _time(lambda i: nat.attention(qkv[i], out[i], B, N, heads, dh,
                                                            dropout=(p, 1234 + i) if p > 0 else None), nbuf, reps)


def linear_case(M, K, N, nbuf=2):
    """x + gamma (W y + b) with the fp32 residual stream (proj: K = E, fc2: K = 4 E)."""
    y = [(torch.randn(M, K, device="cuda") * 0.5).bfloat16() for _ in range(nbuf)]
    w = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
    g, b = torch.full((N,), 0.1, device="cuda"), torch.zeros(N, device="cuda")
    res = [torch.randn(M, N, device="cuda") for _ in range(nbuf)]
    out = [torch.empty(M, N, device="cuda") for _ in range(nbuf)]
    return lambda p, reps=20: _time(lambda i: nat.linear_f32(y[i], w, scale=g, bias=b, res=res[i], res_mode=2, out=out[i],
                                                             dropout=(p, 99 + i) if p > 0 else None), nbuf, reps)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("shape", nargs="*", type=int, help="B N heads dh (default 256 197 12 64)")
    ap.add_argument("--p", type=float, default=0.0, help="attention dropout probability (b200_attention_mc)")
    ap.add_argument("--mc", action="store_true", help="alternate p = 0 / 0.1 over the MC-dropout launches")
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not a.mc:
        B, N, heads, dh = a.shape if len(a.shape) == 4 else (256, 197, 12, 64)
        ms = attention_case(B, N, heads, dh)(a.p)
        flops = 4.0 * B * heads * N * N * dh
        bytes_ = B * N * 4 * heads * dh * 2
        print(f"b200_attention B={B} N={N} heads={heads} dh={dh} p={a.p}: {ms * 1e3:.1f} us/launch, "
              f"{flops / ms / 1e9:.1f} TFLOP/s, {bytes_ / ms / 1e6:.0f} GB/s algorithmic, "
              f"{ms * 1e3 / (B * heads):.2f} us per (case, head) over all SMs")
        return
    print(f"GPU: {gpu_info()}")
    cases = {"attention hybrid (1024, 256, 4 x 128)": attention_case(1024, 256, 4, 128),
             "attention ViT-B/16 (256, 197, 12 x 64)": attention_case(256, 197, 12, 64),
             "proj linear_f32 (262144 x 512 -> 512)": linear_case(1024 * 256, 512, 512),
             "fc2 linear_f32 (262144 x 2048 -> 512)": linear_case(1024 * 256, 2048, 512)}
    times = {k: {0.0: [], 0.1: []} for k in cases}
    for _ in range(a.rounds):
        for k, fn in cases.items():
            for p in (0.0, 0.1):
                times[k][p].append(fn(p))
    for k, t in times.items():
        t0, t1 = min(t[0.0]), min(t[0.1])
        print(f"{k}: p=0 {t0 * 1e3:.1f} us, p=0.1 {t1 * 1e3:.1f} us, ratio {t1 / t0:.2f} "
              f"(best of {a.rounds} rounds of 20 launches; all p=0 {[round(x * 1e3, 1) for x in t[0.0]]}, "
              f"p=0.1 {[round(x * 1e3, 1) for x in t[0.1]]})")


if __name__ == "__main__":
    main()
