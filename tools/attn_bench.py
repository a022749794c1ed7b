"""Stand-alone timing of b200_attention (CUDA events, L2-cold by rotating buffers).

    python tools/attn_bench.py [B N heads dh] [--p P]   one shape; P > 0 times b200_attention_mc (attention dropout)
    python tools/attn_bench.py --mc                      MC-dropout costs: p = 0 and p = 0.1 alternated in one process
                                                         at the hybrid stage (B = 1024, 256 tokens, 4 x 128) and the
                                                         ViT-B/16 shape (B = 256, 197 tokens, 12 x 64), and the proj /
                                                         fc2 launches of linear_f32 (b200_linear vs b200_linear_mc)
    python tools/attn_bench.py --long [--mc]             more than 256 tokens (the key-tiled kernel): ViT-B/16 at
                                                         256 x 256 (B = 256, 257 tokens, 12 x 64), the hybrid stage at
                                                         128 x 128 ROIs (B = 256, 1024 tokens, 4 x 128) and at 256 x 256
                                                         ROIs (B = 64, 4096 tokens, 4 x 128); --mc at p = 0.1.  Beside
                                                         each, torch's scaled_dot_product_attention on the same bf16
                                                         tensors as a yardstick (never on the product path)
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


SUSTAINED_BF16_TFLOPS = 1420.7  # measured sustained dense bf16 peak of the B200 (DESIGN.md section 4)


def sdpa_case(B, N, heads, dh, p, nbuf=4):
    """torch SDPA on the same packed bf16 qkv rows (q, k, v as strided [B, heads, N, dh] views), and the name of the
    kernel it dispatched to (read off one profiled call)."""
    import torch.nn.functional as F
    from torch.profiler import ProfilerActivity, profile

    C = heads * dh
    qkv = [(torch.randn(B * N, 3 * C, device="cuda") * 0.9).bfloat16() for _ in range(nbuf)]
    views = [tuple(t.view(B, N, 3, heads, dh).permute(2, 0, 3, 1, 4)) for t in qkv]
    run = lambda i: F.scaled_dot_product_attention(*views[i], dropout_p=p)
    run(0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(0)
        torch.cuda.synchronize()
    top = max(prof.key_averages(), key=lambda e: getattr(e, "device_time_total", 0.0))
    return (lambda reps=20: _time(run, nbuf, reps)), top.key[:90]


def long_set(mc, rounds):
    p = 0.1 if mc else 0.0
    shapes = {"ViT-B/16 at 256 x 256": (256, 257, 12, 64), "hybrid at 128 x 128 ROIs": (256, 1024, 4, 128),
              "hybrid at 256 x 256 ROIs": (64, 4096, 4, 128)}
    print(f"GPU: {gpu_info()}; attention dropout p = {p}; TFLOP/s of 4 N^2 d heads B; share of the measured sustained "
          f"bf16 peak {SUSTAINED_BF16_TFLOPS} TFLOP/s")
    for name, (B, N, heads, dh) in shapes.items():
        ours = attention_case(B, N, heads, dh)
        ref, backend = sdpa_case(B, N, heads, dh, p)
        t_ours, t_ref = [], []
        for _ in range(rounds):  # alternated in one process
            t_ours.append(ours(p))
            t_ref.append(ref())
        flops = 4.0 * B * heads * N * N * dh
        for tag, t in (("b200_attention" + ("_mc" if mc else ""), t_ours), (f"torch SDPA [{backend}]", t_ref)):
            ms = min(t)
            tf = flops / ms / 1e9
            print(f"{name} (B={B}, N={N}, {heads} x {dh}) {tag}: {ms * 1e3:.1f} us, {tf:.0f} TFLOP/s = "
                  f"{100 * tf / SUSTAINED_BF16_TFLOPS:.1f} % of sustained (best of {rounds} rounds of 20 launches, "
                  f"L2-cold; all {[round(x * 1e3, 1) for x in t]})")
        del ours, ref
        torch.cuda.empty_cache()
    # the third query tile of N = 257 holds one query: the same launch at N = 256 (the one-tile kernel) and N = 384
    # (three full query tiles through the key-tiled kernel) bracket what that tile costs
    for N in (256, 384):
        fn = attention_case(256, N, 12, 64)
        print(f"ViT-B/16 shape at N = {N}: {min(fn(p) for _ in range(rounds)) * 1e3:.1f} us")
        del fn
        torch.cuda.empty_cache()


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("shape", nargs="*", type=int, help="B N heads dh (default 256 197 12 64)")
    ap.add_argument("--p", type=float, default=0.0, help="attention dropout probability (b200_attention_mc)")
    ap.add_argument("--mc", action="store_true", help="alternate p = 0 / 0.1 over the MC-dropout launches")
    ap.add_argument("--long", action="store_true", help="the shapes above 256 tokens, against torch SDPA")
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if a.long:
        long_set(a.mc, a.rounds)
        return
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
