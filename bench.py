#!/usr/bin/env python
"""Benchmark of the hot path: fused DWI+DCE classification, cases/sec (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--aux full|logits]
    python bench.py --impl reference ...      # the reference algorithm on the host CPU cores
    python bench.py --workload c4|resnet       # ViT-B/16 / ResNet-50 backbone encoders at 224x224 (not the headline)
    python bench.py --workload c5 [--encoders c4] [--objective cls]   # fusion-head fine-tuning step (forward +
                                               # backward + gradient all-reduce + AdamW), its own metric line

Workload (BASELINE.json configs[2], the configuration the metric "fused DWI+DCE classify" is
quoted on): per step one batch of B synthetic cases per GPU - raw DWI [B,16,64,64] and DCE
[B,6,64,64] fp32 -> DWINormalize / Nyul -> DWI and DCE CNN encoders -> FusionModel -> logits.
Weights are seeded random (no checkpoints offline), all API outputs are materialised
("aux": "full") unless --aux logits.

One JSON line on stdout (rank 0).  `value`: device-resident inputs, CUDA-event timed, max over
ranks.  `e2e`: the same through FusionPipeline.classify_host with pinned host inputs uploaded
and logits read back every step.  `roofline`: the dominant kernel (3x3 256->256 implicit-GEMM
convolution) timed per launch with CUDA events during a repeat of the timed steps.
`cpu_baseline`: oracle/ (the CPU restatement of the reference) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1; rank 0 also times the CPU reference arm, which must see every host core
if os.environ.get("OMP_NUM_THREADS") == "1" and os.environ.get("RANK", "0") == "0":
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

import torch  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import b200path  # noqa: E402,F401

METRIC = "fused DWI+DCE classify cases/sec"
UNIT = "cases/s"
WORKLOAD = "C3: DWI 16x64x64 + DCE 6x64x64 -> normalise -> CNN encoders -> late-fusion head"
FLOP_PER_CASE_FULL = 9.418e9    # SURVEY.md section 8(d): observable graph, all API outputs
FLOP_PER_CASE_LOGITS = 5.37e9   # logit path only
# --workload c4 (not the default line): the ViT-B/16 backbone configuration of BASELINE.json configs[3]
WORKLOAD_C4 = ("C4: DWI 16x64x64 + DCE 6x64x64 -> resize 224 -> normalise -> ViT-B/16 + adapter encoders -> "
               "late-fusion head")
WORKLOAD_RESNET = ("DWI 16x64x64 + DCE 6x64x64 -> resize 224 -> normalise -> ResNet-50 (output stride 8) + adapter "
                   "encoders -> late-fusion head")
FLOP_RESNET = 116.9e9   # per case, observable graph: hook count on the reference modules (58.6 + 57.8 + 0.84 GF) minus the dead fusion branch
FLOP_C4_FULL = 148.8e9          # SURVEY.md section 8(d)
FLOP_C4_LOGITS = 138.6e9


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tf_burst": p["bf16_tflops"], "tf_sustained": p["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons of this rank's GPU while the timed region runs: NVML in-process
    (10 ms period, so even a 0.2 s region gets ~20 samples), `nvidia-smi -lms` as the fallback."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASON_BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None
        self.stop = threading.Event()
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            props = torch.cuda.get_device_properties(index)
            try:
                bus = f"{props.pci_domain_id:08x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
                self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll_nvml(self):
        n = self.nvml
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        while not self.stop.is_set():
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append([str(sm), str(mx)] + ["Active" if bits & b else "Not Active"
                                                       for b in (0x8, 0x40, 0x20, 0x4)])
            except Exception:
                pass
            self.stop.wait(0.01)

    def __enter__(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        self.stop.set()
        if self.proc is not None:
            self.proc.terminate()
        if self.thread is not None:
            self.thread.join(timeout=2)

    def summary(self):
        sm = [int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------ data ----
def make_inputs(batch, rank):
    g = torch.Generator().manual_seed(1234 + rank)
    dwi = torch.rand(batch, 16, 64, 64, generator=g) * 1000.0 + 1.0
    dce = torch.rand(batch, 6, 64, 64, generator=g)
    dce = dce / dce.amax(dim=(1, 2, 3), keepdim=True)  # prepare_single_model.py:338-339
    return dwi, dce


def make_params(workload, hybrid=False):
    """Parameter dict (+ backbones for c4, configured as foundation_model.build_medical_backbone does)."""
    import parameters_default as pd

    if workload == "c3":
        params = pd.default_parameters()
        for m in ("dwi", "dce"):
            params[f"{m}_model_parameters"]["use_hybrid_transformer"] = hybrid
        return params, {"dwi": None, "dce": None}
    import foundation_model as fm

    params = pd.default_parameters(input_size=224)
    backbones = {}
    for m, c in (("dwi", 16), ("dce", 6)):
        mp = params[f"{m}_model_parameters"]
        mp["backbone_str"], mp["use_backbone"] = ("vit_base_patch16_224" if workload == "c4" else "radimagenet"), True
        backbones[m] = fm.build_medical_backbone(params, None, m, in_channels=c)
    if workload == "c4":
        fs = params["fusion_model_parameters"]["fusion_specific_parameters"]
        fs["dwi_out_channels"] = fs["dce_out_channels"] = 768  # SURVEY.md note 9: not updated by the reference itself
    return params, backbones


def build_product(device, aux, hybrid=False, workload="c3"):
    import model_module as mm
    import parameters_default as pd
    import preprocess_helpers as pre
    from pipeline import FusionPipeline

    torch.manual_seed(0)  # before make_params: the c4 / resnet backbones draw their weights there
    params, backbones = make_params(workload, hybrid)
    mods = [mm.initialize_model(mm.ModelMaskHeadBackbone("dwi", params, backbones["dwi"]), True),
            mm.initialize_model(mm.ModelMaskHeadBackbone("dce", params, backbones["dce"]), True),
            mm.initialize_model(mm.FusionModel(params), True)]
    g = torch.Generator().manual_seed(1)
    for m in mods:  # randomise BN running stats so BN folding is exercised (SURVEY.md section 8d)
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.copy_(0.1 * torch.randn(mod.running_mean.shape, generator=g))
                mod.running_var.copy_(0.5 + torch.rand(mod.running_var.shape, generator=g))
    cpu_state = [{k: v.clone() for k, v in m.state_dict().items()} for m in mods]
    for m in mods:
        m.to(device).eval()
    _, fit_dce = make_inputs(64, 10_000)
    nyul = pre.NyulStandardizer()
    nyul.fit(list(fit_dce), num_channels=6)
    if workload != "c3":  # the standardiser sees resized images (Resize comes first in the reference's transforms)
        from dataset import Resize
        nyul = pre.NyulStandardizer()
        nyul.fit(list(Resize(224).batch(fit_dce[:16].to(device)).cpu()), num_channels=6)
    pipe = FusionPipeline(mods[0], mods[1], mods[2], nyul, aux_mode=aux,
                          input_size=224 if workload != "c3" else None).eval()
    return params, pipe, cpu_state, nyul


DUMP_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """--dump-outputs: {name: tensor} -> directory/<name>.npy, float32.  When the arrays exceed DUMP_BYTES together,
    every one is cut to the same fixed stride of its flattened elements, so repeated runs store the same sample."""
    import numpy as np

    arrays = {k: v.detach().float() for k, v in arrays.items()}
    total = sum(v.numel() for v in arrays.values()) * 4
    stride = -(-total // DUMP_BYTES)
    os.makedirs(directory, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), (v if stride == 1 else v.reshape(-1)[::stride]).cpu().numpy())


def flat_parameters(params):
    return torch.cat([q.detach().float().reshape(-1) for q in params])


# --------------------------------------------------------------------- CPU baseline ----
def cpu_reference_step(params, cpu_state, landmarks, dwi, dce):
    """One batch through oracle/ (CPU restatement of the reference path, incl. its dead fusion branch)."""
    from oracle import model_oracle as mo
    from oracle import normalize_oracle as no

    with torch.no_grad():
        if params["dwi_model_parameters"]["use_backbone"]:  # C4: Resize(224) ahead of the normalisers
            dwi, dce = no.resize(dwi, 224), no.resize(dce, 224)
        x_d = no.dwi_normalize_batch(dwi)
        x_c = no.nyul_transform_batch(dce, landmarks)
        sds = {"dwi": cpu_state[0], "dce": cpu_state[1], "fusion": cpu_state[2]}
        return mo.pipeline_forward(sds, params, x_d, x_c, run_dead_branch=True)[0]


def run_cpu_baseline(params, cpu_state, nyul, cases, batch, warmup_batches=1):
    import numpy as np

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    lm = np.stack([nyul.channel_landmarks[c] for c in range(6)])
    dwi, dce = make_inputs(batch, 777)
    for _ in range(warmup_batches):
        cpu_reference_step(params, cpu_state, lm, dwi, dce)
    n_batches = max(1, cases // batch)
    t0 = time.perf_counter()
    for _ in range(n_batches):
        cpu_reference_step(params, cpu_state, lm, dwi, dce)
    dt = time.perf_counter() - t0
    return {"value": n_batches * batch / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_batches} batches of {batch} cases of the same workload, fp32, torch CPU threads={threads}, "
                      f"1 warm-up batch, {dt:.1f} s"}


def reference_arm(args):
    """--impl reference: the reference algorithm (oracle port; the Python reference itself cannot travel
    to the GPU box) on the host cores, same metric/config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import model_module as mm  # parameter containers only (state_dict source); no CUDA needed
    import parameters_default as pd
    import preprocess_helpers as pre
    import numpy as np

    params, backbones = make_params(args.workload)
    torch.manual_seed(0)
    mods = [mm.initialize_model(mm.ModelMaskHeadBackbone("dwi", params, backbones["dwi"]), True),
            mm.initialize_model(mm.ModelMaskHeadBackbone("dce", params, backbones["dce"]), True),
            mm.initialize_model(mm.FusionModel(params), True)]
    cpu_state = [m.state_dict() for m in mods]
    _, fit_dce = make_inputs(64, 10_000)
    if args.workload != "c3":
        from oracle import normalize_oracle as no
        fit_dce = no.resize(fit_dce[:16], 224)
    nyul = pre.NyulStandardizer()
    nyul.fit(list(fit_dce), num_channels=6)
    lm = np.stack([nyul.channel_landmarks[c] for c in range(6)])
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    batch = args.ref_batch
    dwi, dce = make_inputs(batch, 777)
    for _ in range(args.warmup):
        cpu_reference_step(params, cpu_state, lm, dwi, dce)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_step(params, cpu_state, lm, dwi, dce)
    dt = time.perf_counter() - t0
    value = args.steps * batch / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": {"c3": WORKLOAD, "c4": WORKLOAD_C4, "resnet": WORKLOAD_RESNET}[args.workload], "batch_per_step": batch,
                   "aux": "full (as the reference executes)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"each step = {batch} cases (reference batch_size) of the workload on {threads} host threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))



def gemm_flops(name, key):
    """2*M*N*K of a GEMM-shaped launch from its profile key (None for everything else)."""
    if key is None:
        return None
    if name == "b200_conv_gemm_ex":      # (B, H, W, Cin, Cout, taps)
        b_, h_, w_, ci, co, tp = key[:6]
        st = 2 if tp == 4 else (key[6] if len(key) > 6 else 1)
        return 2.0 * b_ * (h_ * w_ // (st * st)) * ci * co * tp
    if name == "b200_linear":            # (M, K, N)
        return 2.0 * key[0] * key[1] * key[2]
    if name == "b200_gemm_batched":      # (batch, heads, M, K, N, mode)
        return 2.0 * key[0] * key[1] * key[2] * key[3] * key[4]
    return None


# --------------------------------------------------------------- fusion-head fine-tuning (C5 slice) ----
WORKLOAD_C5 = ("C5 (frozen-encoder phase): DWI 16x64x64 + DCE 6x64x64 -> normalise -> frozen CNN encoders -> "
               "fusion-head forward + backward (smoothed focal loss + mask dice) -> gradient all-reduce -> AdamW")
METRIC_C5 = "fusion-head fine-tuning cases/sec"


def train_arm(args):
    """--workload c5: one optimisation step of the fusion head per batch (fusion_train.FusionHeadTrainer), data
    parallel over the ranks with ONE NCCL all-reduce of the flat gradient buffer per step."""
    import b200_native as nat
    from fusion_train import FusionHeadTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import datetime
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    enc = args.encoders
    params, pipe, cpu_state, nyul = build_product(device, "logits", False, enc)
    lam = 0.2 if args.objective == "cls+mask" else 0.0   # lambda_mask, parameters_generate.py:125
    trainer = FusionHeadTrainer(pipe.fusion_model, lr=1e-4, weight_decay=4e-5, smoothing=0.1, gamma=1.5,
                                lambda_mask=lam)
    B = args.batch
    dwi_h, dce_h = make_inputs(B, rank)
    gen = torch.Generator().manual_seed(99 + rank)
    lab_h = torch.randint(0, 4, (B,), generator=gen)
    msk_h = (torch.rand(B, 1, 32, 32, generator=gen) > 0.5).float()
    dwi_d, dce_d, lab_d, msk_d = dwi_h.to(device), dce_h.to(device), lab_h.to(device), msk_h.to(device)

    def step():
        loss, _ = trainer.train_step(*pipe.encode_raw(dwi_d, dce_d), lab_d, msk_d if lam > 0 else None)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = nat.LAUNCH_COUNT
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        torch.cuda.nvtx.range_push("timed")  # ncu --nvtx --nvtx-include "timed/" captures exactly these steps
        e0.record()
        for _ in range(args.steps):
            loss = step()
        e1.record()
        barrier()
        torch.cuda.nvtx.range_pop()
    launches = nat.LAUNCH_COUNT - launches0
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss.reshape(1),
                                         "fusion_parameters": flat_parameters(pipe.fusion_model.parameters())})
    ms = e0.elapsed_time(e1)
    # end to end: pinned host batch (inputs + labels) uploaded every step, the loss read back every step
    dwi_p, dce_p, lab_p, msk_p = dwi_h.pin_memory(), dce_h.pin_memory(), lab_h.pin_memory(), msk_h.pin_memory()
    host_batch = (dwi_p, dce_p, lab_p, msk_p) if lam > 0 else (dwi_p, dce_p, lab_p)
    pipe.fit_host([host_batch] * 2, trainer)
    barrier()
    e0.record()
    pipe.fit_host([host_batch] * args.steps, trainer)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = t[0].item(), t[1].item()
    value = world * B * args.steps / (ms / 1e3)
    # data-parallel invariant: after the same number of steps every replica holds bit-identical parameters
    in_sync = True
    if world > 1:
        flat_p = trainer._bind()["p"]
        lo, hi = flat_p.clone(), flat_p.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        in_sync = bool(torch.equal(lo, hi))
    line = None
    if rank == 0:
        peaks = load_peaks()
        nsp = max(2, min(args.steps, 5))
        nat.start_profile()
        for _ in range(nsp):
            step() if world == 1 else None
        prof = nat.stop_profile()
        total_ms = sum(sum(t) for t in prof.values())
        head = {n: 0.0 for n in ("b200_sgemm", "b200_colsum", "b200_mha_fwd", "b200_mha_bwd", "b200_ln_fwd",
                                 "b200_ln_bwd", "b200_gelu_bwd", "b200_head_loss", "b200_adamw", "b200_fusion_tokens",
                                 "b200_mask_dot", "b200_mask_wsum", "b200_mask_dice", "b200_mask_head_grads")}
        sg_flops = sg_ms = 0.0
        for (n, k), t in prof.items():
            if n in head:
                head[n] += sum(t) / nsp
            if n == "b200_sgemm" and k is not None:
                sg_flops += 2.0 * k[0] * k[1] * k[2] * len(t) / nsp
                sg_ms += sum(t) / nsp
        # the map-sized passes of the head are HBM bound: algorithmic bytes = one read of the bf16 f3 map per launch
        hbm_rows = []
        f3_shape = (32, 32, 512) if enc == "c3" else (14, 14, 768)
        f3_bytes = B * f3_shape[0] * f3_shape[1] * f3_shape[2] * 2
        # dram__bytes_read.sum + dram__bytes_write.sum per launch at B = 1024 (profiles/r1_c5_hbm_kernels_ncu.csv)
        ncu_traffic = {"b200_fusion_tokens": 1.0738e9 + 32.3e6, "b200_mask_dot": 1.0758e9 + 9.0e6}
        for n in ("b200_fusion_tokens", "b200_mask_dot", "b200_mask_wsum"):
            times = [x for (nn_, _), t in prof.items() if nn_ == n for x in t]
            if times:
                ms_l = statistics.mean(times)
                gbs = f3_bytes / (ms_l / 1e3) / 1e9
                hbm_rows.append({"bound": "hbm", "kernel": n, "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": gbs / peaks["hbm_gbs"], "ms_per_launch": ms_l,
                                 "traffic": ncu_traffic[n] * B / 1024 if n in ncu_traffic and enc == "c3" else None,
                                 "algorithmic_bytes_per_launch": f3_bytes})
        if enc == "c3":
            dom_key = ("b200_conv_gemm_ex", (B, 32, 32, 256, 256, 9))
            dom_name = "conv_gemm_kernel<256> 3x3 256->256 @32x32 (frozen encoders: still the dominant launch)"
        else:  # the GEMM-shaped launch class with the largest share of the step
            cands = [(sum(t), nk) for nk, t in prof.items() if gemm_flops(*nk) is not None]
            dom_key = max(cands)[1] if cands else None
            dom_name = f"conv_gemm_kernel via {dom_key[0]} {list(dom_key[1])} (frozen encoders)" if dom_key else None
        roofline = None
        if dom_key in prof:
            dom_ms = statistics.mean(prof[dom_key])
            ach = gemm_flops(*dom_key) / (dom_ms / 1e3) / 1e12
            roofline = {"bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                        "frac": ach / peaks["tf_sustained"], "traffic": 1.032e9 * B / 1024 if enc == "c3" else None,
                        "kernel": dom_name,
                        "ms_per_launch": dom_ms, "share_of_step": sum(prof[dom_key]) / total_ms if total_ms else None,
                        "peak_source": peaks["source"] + " sustained bf16"}
        line = {
            "metric": METRIC_C5, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 encoders (frozen) / f32 head forward, backward and optimiser",
            "data": "synthetic",
            "config": {"workload": WORKLOAD_C5 if enc == "c3" else WORKLOAD_C5.replace(
                           "normalise -> frozen CNN encoders", "resize 224 -> normalise -> frozen ViT-B/16 + adapter encoders"),
                       "batch_per_gpu": B, "global_batch": B * world,
                       "objective": "classification (label smoothing 0.1, focal gamma 1.5)" +
                       (" + 0.2 x mean of the three mask dice terms" if lam > 0 else " only"),
                       "trainable_parameters": trainer.numel, "allreduce_bytes_per_step": 4 * (trainer.flat_numel + 1),
                       "l2": "no flush needed: per-step inputs and activations exceed the 126 MB L2",
                       "parallelism": f"data parallel x{world}, one NCCL all-reduce of the flat gradient buffer per step"
                       if world > 1 else "single GPU"},
            "clocks": clocks.summary(),
            "e2e": {"value": world * B * args.steps / (e2e_ms / 1e3), "unit": UNIT,
                    "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host_batch),
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / args.steps,
                    "api": "FusionPipeline.fit_host (pinned host batch incl. labels, upload overlapped on a copy stream, "
                    "loss read back every step)"},
            "gpu_launches": launches, "final_loss": float(loss.item()), "replicas_in_sync": in_sync,
            "hbm_peak_allocated_gb": torch.cuda.max_memory_allocated(device) / 1e9,
            "roofline": roofline,
            "roofline_hbm_kernels": hbm_rows,
            "step_model": {"head_kernels_ms_per_step": {k: round(v, 4) for k, v in head.items()},
                           "head_share_of_step": sum(head.values()) / (total_ms / nsp) if total_ms else None,
                           "sgemm_fp32_tflops": sg_flops / (sg_ms / 1e3) / 1e12 if sg_ms else None},
            "cpu_baseline": None,
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = (run_cpu_train_baseline(params, cpu_state, nyul, args.ref_batch, lam)
                                    if enc == "c3" else None)  # (the C4 CPU forward alone is ~1 s per case)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# --workload c5 --unfrozen / --objective full, and --workload c1: the training step on the training kernels
# ------------------------------------------------------------------------------------------------------------------
WORKLOAD_C5_FULL = ("C5: fusion fine-tuning step, backbone (both CNN encoders) UNFROZEN, bf16 activations and gradient maps, "
                    "fp32 master weights: normalise -> train-mode DWI / DCE encoders + fusion head (batch-statistic "
                    "BatchNorm, dropout 0.2) -> classification + 3 dice + 3 reconstruction + mimic terms -> explicit "
                    "backward (dgrad / wgrad on tcgen05) -> bucketed NCCL gradient all-reduce -> fused AdamW")
WORKLOAD_C1 = ("C1: DWI-only model_module CNN forward + train step on synthetic 16-b-value 64x64 ROIs, batch 32 "
               "(LightningSingleModel._shared_step objective: classification + feature norm + mask dice + reconstruction "
               "+ mimic) -> backward -> AdamW")


def _train_flops_per_case(unfrozen):
    """Algorithmic FLOPs of one training step per case: forward of the graph that is evaluated + dgrad + wgrad of every
    convolution whose input / weight needs a gradient (2 MAC = 2 FLOP).  Encoder logit-path + reconstruction heads
    (no encoder classifier / projectors in the fusion step): 4.06 GF forward per encoder (SURVEY 8a: 4.40 minus
    0.34 of projectors); fusion head 0.616 GF.  Training = 3x the forward of everything trainable (the stem's data
    gradient is not needed, < 0.1 %)."""
    enc = 4.06e9
    fus = 0.616e9
    return 3 * (2 * enc + fus) if unfrozen else (2 * 2.545e9 + 3 * fus)


def train_full_arm(args):
    """--workload c5 --unfrozen (BASELINE configs[4]) or --objective full with frozen encoders: one optimisation step per
    batch on train_graph.FullFusionTrainer."""
    import b200_native as nat
    import train_graph as tg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import datetime
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    unfrozen = bool(args.unfrozen)
    params, pipe, cpu_state, nyul = build_product(device, "logits", False, "c3")
    for m in (pipe.dwi_model, pipe.dce_model, pipe.fusion_model):
        for q in m.parameters():
            q.requires_grad_(True)
        m.train() if (unfrozen or m is pipe.fusion_model) else m.eval()
    trainer = tg.FullFusionTrainer(pipe.dwi_model, pipe.dce_model, pipe.fusion_model, lr=1e-4, weight_decay=4e-5,
                                   smoothing=0.1, gamma=1.5, lambda_mask=0.2, lambda_recon=0.1, lambda_mimic=0.2,
                                   encoders_trainable=unfrozen)
    B = args.batch
    dwi_h, dce_h = make_inputs(B, rank)
    gen = torch.Generator().manual_seed(99 + rank)
    lab_h = torch.randint(0, 4, (B,), generator=gen)
    msk_h = (torch.rand(B, 1, 32, 32, generator=gen) > 0.5).float()
    dwi_d, dce_d, lab_d, msk_d = dwi_h.to(device), dce_h.to(device), lab_h.to(device), msk_h.to(device)

    def step_on(dwi_raw, dce_raw, lab, msk):
        dwi = pipe.dwi_norm.batch(dwi_raw)
        dce = pipe.dce_norm.batch(dce_raw)
        if unfrozen:
            return trainer.train_step(dwi, dce, msk, lab)[0]
        with torch.no_grad():
            o_d = pipe.dwi_model(dwi, None)
            o_c = pipe.dce_model(dce, None)
        f3d = o_d[1]["raw_feats"][-1].permute(0, 2, 3, 1)
        f3c = o_c[1]["raw_feats"][-1].permute(0, 2, 3, 1)
        return trainer.train_step(dwi, dce, msk, lab, md=o_d[2][:, 0].contiguous(), mc=o_c[2][:, 0].contiguous(),
                                  f3d=f3d, f3c=f3c)[0]

    def step():
        return step_on(dwi_d, dce_d, lab_d, msk_d)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = nat.LAUNCH_COUNT
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        torch.cuda.nvtx.range_push("timed")
        e0.record()
        for _ in range(args.steps):
            loss = step()
        e1.record()
        barrier()
        torch.cuda.nvtx.range_pop()
    launches = nat.LAUNCH_COUNT - launches0
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss.reshape(1), "trained_parameters": flat_parameters(trainer.params)})
    ms = e0.elapsed_time(e1)
    # end to end: pinned host batch uploaded every step (copy stream, overlapped with the previous step), loss read back
    host_batch = tuple(t.pin_memory() for t in (dwi_h, dce_h, lab_h, msk_h))

    def fit_host(n):
        losses = []
        for d, c, lab, msk in pipe._staged([host_batch] * n, device):
            l_ = step_on(d, c, lab, msk)
            h = torch.empty(1, dtype=torch.float32, pin_memory=True)
            h.copy_(l_, non_blocking=True)
            losses.append(h)
        torch.cuda.current_stream(device).synchronize()
        return losses

    fit_host(2)
    barrier()
    e0.record()
    fit_host(args.steps)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = t[0].item(), t[1].item()
    value = world * B * args.steps / (ms / 1e3)
    in_sync = True
    if world > 1:
        lo, hi = trainer.flat["p"].clone(), trainer.flat["p"].clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        in_sync = bool(torch.equal(lo, hi))
    line = None
    if rank == 0:
        peaks = load_peaks()
        nsp = 2
        prof = {}
        if world == 1:
            nat.start_profile()
            for _ in range(nsp):
                step()
            prof = nat.stop_profile()
        total_ms = sum(sum(t) for t in prof.values())
        by_name = {}
        for (n, k), t in prof.items():
            by_name[n] = by_name.get(n, 0.0) + sum(t) / nsp
        # dominant launches: forward / data-gradient GEMMs (b200_conv_gemm_ex) and the weight-gradient kernel
        roofline = None
        wg = [(sum(t), t) for (n, k), t in prof.items() if n == "b200_conv_wgrad"]
        cands = [(sum(t), nk) for nk, t in prof.items() if gemm_flops(*nk) is not None]
        if cands:
            dom_key = max(cands)[1]
            dom_ms = statistics.mean(prof[dom_key])
            ach = gemm_flops(*dom_key) / (dom_ms / 1e3) / 1e12
            roofline = {"bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                        "frac": ach / peaks["tf_sustained"], "frac_of_burst_peak": ach / peaks["tf_burst"], "traffic": None,
                        "kernel": f"conv_gemm_kernel via {dom_key[0]} {list(dom_key[1])} (forward and data-gradient launches "
                                  "of this shape)", "ms_per_launch": dom_ms,
                        "share_of_step": sum(prof[dom_key]) / total_ms if total_ms else None,
                        "peak_source": peaks["source"] + " sustained bf16"}
        flop_case = _train_flops_per_case(unfrozen)
        line = {
            "metric": METRIC_C5, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16 activations / gradient maps, fp32 accumulation, master weights and optimiser", "data": "synthetic",
            "config": {"workload": WORKLOAD_C5_FULL if unfrozen else WORKLOAD_C5_FULL.replace(
                           "backbone (both CNN encoders) UNFROZEN", "frozen-encoder phase (eval-mode encoders), full objective"),
                       "batch_per_gpu": B, "global_batch": B * world, "trainable_parameters": trainer.numel,
                       "allreduce_bytes_per_step": 4 * (trainer.flat_numel + 1),
                       "allreduce_buckets": "cut at block boundaries in backward order, >= 8 MB each, issued on a side "
                                            "stream while the rest of the backward pass runs",
                       "l2": "no flush needed: per-step inputs and activations exceed the 126 MB L2",
                       "parallelism": f"data parallel x{world} (NCCL)" if world > 1 else "single GPU"},
            "clocks": clocks.summary(),
            "e2e": {"value": world * B * args.steps / (e2e_ms / 1e3), "unit": UNIT,
                    "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host_batch), "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / args.steps,
                    "api": "pinned host batch (raw ROIs, labels, target masks) -> FusionPipeline normalisers -> "
                           "FullFusionTrainer.train_step, upload overlapped on a copy stream, loss read back every step"},
            "gpu_launches": launches, "final_loss": float(loss.item()), "replicas_in_sync": in_sync,
            "hbm_peak_allocated_gb": torch.cuda.max_memory_allocated(device) / 1e9,
            "roofline": roofline,
            "step_model": {"algorithmic_gflop_per_case": flop_case / 1e9,
                           "achieved_tflops_whole_step": value / world * flop_case / 1e12,
                           "frac_of_sustained_peak": value / world * flop_case / 1e12 / peaks["tf_sustained"],
                           "ms_per_step_by_entry_point": {k: round(v, 3) for k, v in sorted(by_name.items(), key=lambda kv: -kv[1])},
                           "wgrad_launches_ms": round(sum(s for s, _ in wg) / nsp, 3) if wg else None},
            "cpu_baseline": None,
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))


def c1_arm(args):
    """--workload c1 (BASELINE configs[0]): DWI CNN forward + train step at batch 32 - on the GPU through
    train_graph (forward, single-model objective, backward, AdamW) and, beside it, the reference's CPU path (oracle
    restatement of LightningSingleModel._shared_step + backward + AdamW, pinned by tests/golden/train_c1_dwi.npz) on the
    host cores."""
    import b200_native as nat
    import model_module as mm
    import parameters_default as pd
    import train_graph as tg
    from oracle import params as op
    from oracle import train_oracle as to

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    device = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    B = args.batch
    p = pd.default_parameters()
    model = mm.ModelMaskHeadBackbone("dwi", p)
    sd = op.seeded_state_dict(op.shapes_of(model.state_dict()), seed=7)
    model.load_state_dict(sd)
    model.to(device).train()
    for q in model.parameters():
        q.requires_grad_(True)
    lam = dict(lambda_mask=0.2, lambda_recon=0.1, lambda_mimic=0.2, lambda_feat_norm=4e-5)
    tr = tg.SingleModelTrainer(model, lr=1e-4, weight_decay=4e-5, smoothing=0.1, gamma=1.5, **lam)
    dwi_raw, _, masks, labels = op.synthetic_raw(B, seed=1234, kind="S")
    x_h = (dwi_raw / dwi_raw.amax(dim=(1, 2, 3), keepdim=True)).pin_memory()
    x_d, m_d, l_d = x_h.to(device), masks.to(device), labels.to(device)
    for _ in range(args.warmup):
        tr.train_step(x_d, m_d, l_d)
    torch.cuda.synchronize()
    l0 = nat.LAUNCH_COUNT
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            loss = tr.train_step(x_d, m_d, l_d)[0]
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = nat.LAUNCH_COUNT - l0
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, {"loss": loss.reshape(1), "dwi_parameters": flat_parameters(model.parameters())})
    m_h, l_h = masks.pin_memory(), labels.pin_memory()
    e0.record()
    for _ in range(args.steps):
        loss_h = tr.train_step(x_h.to(device, non_blocking=True), m_h.to(device, non_blocking=True),
                               l_h.to(device, non_blocking=True))[0].cpu()
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1)
    # the reference's CPU path: same batch, same seeded weights
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cw = None
    pc = pd.default_parameters()

    def cpu_step(state, mom, it):
        _, _, grads = to.single_model_objective_and_grads(state, pc, "dwi", x_h, masks, labels, 0.1, 1.5, cw, **lam)
        for k, g in grads.items():
            mm_, vv_ = mom.get(k, (torch.zeros_like(g), torch.zeros_like(g)))
            state[k], mm_, vv_ = to.adamw_step(state[k], g, mm_, vv_, it, 1e-4, (0.9, 0.999), 1e-8, 4e-5)
            mom[k] = (mm_, vv_)

    state, mom = {k: v.clone() for k, v in sd.items()}, {}
    cpu_step(state, mom, 1)
    n_cpu = 3
    t0 = time.perf_counter()
    for it in range(n_cpu):
        cpu_step(state, mom, it + 2)
    dt = time.perf_counter() - t0
    peaks = load_peaks()
    flop_case = 3 * 4.403e9
    value = B * args.steps / (ms / 1e3)
    line = {
        "metric": "DWI CNN train-step cases/sec", "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16 activations / gradient maps, fp32 master weights", "data": "synthetic",
        "config": {"workload": WORKLOAD_C1, "batch_per_gpu": B, "global_batch": B, "trainable_parameters": tr.numel,
                   "note": "batch 32 is the reference's CPU-runnable case: a launch-latency-bound size on a B200 "
                           f"({launches // max(args.steps, 1)} launches per step)"},
        "clocks": clocks.summary(),
        "e2e": {"value": B * args.steps / (e2e_ms / 1e3), "unit": UNIT,
                "h2d_bytes_per_step": x_h.numel() * 4 + m_h.numel() * 4 + l_h.numel() * 8, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms / args.steps, "api": "SingleModelTrainer.train_step on pinned host tensors, loss read back"},
        "gpu_launches": launches, "final_loss": float(loss.item()),
        "roofline": None,
        "step_model": {"algorithmic_gflop_per_case": flop_case / 1e9, "achieved_tflops_whole_step": value * flop_case / 1e12,
                       "frac_of_sustained_peak": value * flop_case / 1e12 / peaks["tf_sustained"]},
        "cpu_baseline": {"value": n_cpu * B / dt, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n_cpu} optimisation steps of {B} cases (forward + backward + AdamW), fp32, torch CPU "
                                   f"threads={threads}, 1 warm-up step, {dt:.1f} s"},
    }
    print(json.dumps(line))


def run_cpu_train_baseline(params, cpu_state, nyul, batch, lambda_mask=0.0, steps=3):
    """The same step on the host cores: oracle encoders (eval, no grad) + oracle/train_oracle.py (autograd over the
    full-resolution FusionModel forward + AdamW)."""
    import numpy as np
    from oracle import model_oracle as mo
    from oracle import normalize_oracle as no
    from oracle import train_oracle as to

    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    lm = np.stack([nyul.channel_landmarks[c] for c in range(6)])
    dwi, dce = make_inputs(batch, 777)
    gen = torch.Generator().manual_seed(5)
    labels = torch.randint(0, 4, (batch,), generator=gen)
    masks = (torch.rand(batch, 1, 32, 32, generator=gen) > 0.5).float()
    sd = {k: v.clone() for k, v in cpu_state[2].items()}

    def one(sd):
        with torch.no_grad():
            x_d, x_c = no.dwi_normalize_batch(dwi), no.nyul_transform_batch(dce, lm)
            _, aux_d, m_d = mo.encoder_forward(cpu_state[0], "dwi", params, x_d)
            _, aux_c, m_c = mo.encoder_forward(cpu_state[1], "dce", params, x_c)
        b = (aux_d["raw_feats"][-1], aux_c["raw_feats"][-1], m_d, m_c, labels)
        return to.train_steps(sd, params, b, 1, 0.1, 1.5, None, 1e-4, (0.9, 0.999), 1e-8, 4e-5, masks, lambda_mask)[1]

    sd = one(sd)
    t0 = time.perf_counter()
    for _ in range(steps):
        sd = one(sd)
    dt = time.perf_counter() - t0
    return {"value": steps * batch / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{steps} optimisation steps of {batch} cases, fp32, torch CPU threads={threads}, 1 warm-up step, "
                      f"{dt:.1f} s"}

# ------------------------------------------------------------------------- B200 arm ----
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="cases per GPU per step (default 1024; 256 for c4)")
    ap.add_argument("--unfrozen", action="store_true",
                    help="--workload c5: BASELINE configs[4] proper - both CNN encoders train too (train-mode BatchNorm, "
                         "dropout, dgrad / wgrad on the tensor cores, bucketed all-reduce); implies --objective full")
    ap.add_argument("--workload", default="c3", choices=["c3", "c4", "resnet", "c5", "c1"],
                    help="c3 = the headline CNN-encoder configuration; c4 = ViT-B/16 backbone encoders at 224x224; "
                         "resnet = ResNet-50 (RadImageNet branch, output stride 8) backbone encoders at 224x224")
    ap.add_argument("--aux", default="full", choices=["full", "logits"])
    ap.add_argument("--encoders", default="c3", choices=["c3", "c4"],
                    help="--workload c5: frozen encoders feeding the head - c3 = the CNN encoders (headline), c4 = "
                         "ViT-B/16 backbone + adapter at 224x224 (768-channel 14x14 maps)")
    ap.add_argument("--objective", default="cls+mask", choices=["cls", "cls+mask", "full"],
                    help="--workload c5: loss terms of the fine-tuning step (the reference's total loss minus its "
                         "reconstruction / mimic terms, or the classification term alone)")
    ap.add_argument("--ref-batch", type=int, default=32)
    ap.add_argument("--cpu-cases", type=int, default=256, help="bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--predict-mode", default="normal", choices=["normal", "tta", "mc", "tta_mc"],
                    help="reference test-time modes (train_fusion.py:682-702); tta_mc = 4 flips x 10 MC-dropout passes, "
                         "the reference's default test_mode.  Not the headline workload.")
    ap.add_argument("--hybrid", action="store_true",
                    help="encoders with the in-house TransformerStage instead of block3 (not the headline workload)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32, at most "
                         "64 MB): the fusion logits of every case, gathered over the ranks (fusion_probabilities in the "
                         "multi-pass predict modes); for c5 / c1 the loss and the parameters after the update.  Inputs "
                         "and weights are seeded, so two builds can be compared output for output; repeated runs of one "
                         "build are close, not bit-identical (the encoders' channel sums are float atomics)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 path")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.workload == "c1":
        args.batch = args.batch or 32
        c1_arm(args)
        return
    if args.batch is None and args.workload == "c5" and (args.unfrozen or args.objective == "full"):
        args.batch = 512
    if args.batch is None:
        args.batch = 1024 if args.workload == "c3" or (args.workload == "c5" and args.encoders == "c3") else 256
    if args.workload not in ("c3", "c5") and args.ref_batch == 32:
        args.ref_batch = 8  # ~1 s per case on the host cores: keep a step / the CPU sample bounded
        args.cpu_cases = min(args.cpu_cases, 16)

    if args.workload == "c5":
        if args.impl == "reference":
            raise SystemExit("--impl reference times the headline inference workload; the c5 line carries its own "
                             "cpu_baseline")
        if args.unfrozen or args.objective == "full":
            train_full_arm(args)
        else:
            train_arm(args)
        return
    if args.impl == "reference":
        reference_arm(args)
        return

    import b200_native as nat

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import datetime
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))

    params, pipe, cpu_state, nyul = build_product(device, args.aux, args.hybrid, args.workload)
    B = args.batch
    dwi_h, dce_h = make_inputs(B, rank)
    dwi_d, dce_d = dwi_h.to(device), dce_h.to(device)

    lightning = None
    if args.predict_mode != "normal":
        import train_fusion as tf_mod
        lightning = tf_mod.LightningFusionModel(pipe.dwi_model, pipe.dce_model, pipe.fusion_model, params)

    def step():
        if lightning is not None:  # normalise once, then the reference's multi-pass prediction mode
            d, c = dwi_d, dce_d
            if pipe.resize is not None:
                d, c = pipe.resize.batch(d), pipe.resize.batch(c)
            d, c = pipe.dwi_norm.batch(d), pipe.dce_norm.batch(c)
            if args.predict_mode == "tta":
                logits = lightning.predict_tta(d, c)[0]
            elif args.predict_mode == "mc":
                logits = lightning.predict_mc_dropout(d, c, passes=10)[0]
            else:
                logits = lightning.predict_tta_mc(d, c, passes=10)[0]
            return logits
        return pipe.forward_raw(dwi_d, dce_d)

    def gather(per_step):
        """The path's only exchange: every rank's logits (16 B/case) collected ONCE for the K steps, inside the timed
        region, as a prediction loop gathers at the end of an epoch (model_test.py:150-163 accumulates per-batch
        predictions and concatenates after the loop) - not a collective per step."""
        if world > 1 and per_step:
            mine = torch.stack(per_step)
            everyone = torch.empty((world,) + tuple(mine.shape), device=device, dtype=mine.dtype)
            dist.all_gather_into_tensor(everyone, mine)
            return everyone
        return None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gather([step() for _ in range(args.warmup)])
    barrier()
    launches0 = nat.LAUNCH_COUNT
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        torch.cuda.nvtx.range_push("timed")  # ncu --nvtx --nvtx-include "timed/" captures exactly these steps
        e0.record()
        per_step = [step() for _ in range(args.steps)]
        gathered = gather(per_step)
        e1.record()
        barrier()
        torch.cuda.nvtx.range_pop()
    launches = nat.LAUNCH_COUNT - launches0
    if args.dump_outputs is not None and rank == 0:
        last = per_step[-1] if gathered is None else gathered[:, -1].reshape(-1, per_step[-1].shape[-1])
        # the multi-pass prediction modes return the mean softmax over their passes, not logits
        dump_outputs(args.dump_outputs, {"fusion_logits" if args.predict_mode == "normal" else "fusion_probabilities": last})
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    value = world * B * args.steps / (ms / 1e3)

    # ---- end-to-end through the public API: pinned host inputs, logits read back ----
    # the pinned buffers are allocated (and the copies issued) from the NUMA node of this rank's GPU
    from sharding import bind_to_device_numa_node, restore_affinity
    numa = bind_to_device_numa_node(local_rank)
    dwi_p, dce_p = dwi_h.pin_memory(), dce_h.pin_memory()
    pipe.classify_host([(dwi_p, dce_p)] * 2)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    outs = pipe.classify_host([(dwi_p, dce_p)] * args.steps)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([e2e_ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = t.item()
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)
    h2d = dwi_p.numel() * 4 + dce_p.numel() * 4
    d2h = outs[0].numel() * 4
    restore_affinity(numa)  # the CPU baseline below uses every host core

    line = None
    if rank == 0:
        peaks = load_peaks()
        # ---- per-launch CUDA-event profile of the same steps (a repeat of the timed region) ----
        nat.start_profile()
        for _ in range(max(2, min(args.steps, 5))):
            pipe.forward_raw(dwi_d, dce_d)  # rank-local: no collective in this rank-0-only pass
        prof = nat.stop_profile()
        table = {}
        total_ms = 0.0
        for (name, key), times in prof.items():
            table[(name, key)] = (statistics.mean(times), len(times))
            total_ms += sum(times)
        if args.workload == "c3":
            dom_key = ("b200_conv_gemm_ex", (B, 32, 32, 256, 256, 9))
            dom_name = "conv_gemm_kernel<256> 3x3 256->256 @32x32"
        else:  # the GEMM-shaped launch class with the largest share of the step
            cands = [(sum(t), nk) for nk, t in prof.items() if gemm_flops(*nk) is not None]
            dom_key = max(cands)[1] if cands else None
            dom_name = f"conv_gemm_kernel via {dom_key[0]} {list(dom_key[1])}" if dom_key else None
        dom_ms, dom_cnt = table.get(dom_key, (None, 0))
        roofline = None
        if dom_ms:
            flops = gemm_flops(*dom_key)
            ach = flops / (dom_ms / 1e3) / 1e12
            # DRAM bytes of this launch from the committed ncu --set full captures (dram__bytes_read.sum +
            # dram__bytes_write.sum, scaled by the batch)
            # profiles/r2_ncu_full.csv: 538 + 494 MB (C3 conv, B = 1024); 82 + 252 MB (C4 fc1, 50 432 rows)
            traffic = 1.032e9 * B / 1024 if args.workload == "c3" else None
            if args.workload == "c4" and dom_key[0] == "b200_conv_gemm_ex" and tuple(dom_key[1][3:]) == (768, 3072, 1):
                traffic = 334.5e6 * dom_key[1][2] / 50432
            roofline = {"bound": "tensor", "achieved": ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                        "frac": ach / peaks["tf_sustained"], "frac_of_burst_peak": ach / peaks["tf_burst"],
                        "traffic": traffic,
                        "traffic_source": ("profiles/r2_ncu_full.csv (r2_conv256): one ncu --set full capture of this kernel "
                                           "(dram__bytes_read.sum + dram__bytes_write.sum), scaled by the batch - a static "
                                           "figure, not re-measured in this run") if traffic is not None else None,
                        "kernel": dom_name,
                        "ms_per_launch": dom_ms, "peak_source": peaks["source"] + " sustained bf16 (the kernel runs inside "
                        "a step of back-to-back GEMM launches; frac_of_burst_peak is against the burst figure)",
                        "share_of_step": sum(prof[dom_key]) / total_ms if total_ms else None}
        # the HBM-bound side of the path: the DWI normaliser against the measured copy bandwidth
        # (algorithmic bytes per case: 15 planes read + 16 written, SURVEY.md section 8(d) / DESIGN.md 4.2)
        hbm_roofline = None
        nm = table.get(("b200_dwi_normalize", None))
        nm_fused = table.get(("b200_dwi_normalize_ex", None))
        side = 224 if args.workload != "c3" else 64
        if nm:
            nbytes = B * (15 + 16) * side * side * 4
            gbs = nbytes / (nm[0] / 1e3) / 1e9
            hbm_roofline = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": gbs / peaks["hbm_gbs"], "traffic": None, "kernel": "dwi_normalize (inside the step)",
                            "ms_per_launch": nm[0], "algorithmic_bytes_per_launch": nbytes}
        fused_norm = None
        if nm_fused:
            # fused first layer (the default for the CNN encoders): the normaliser is a statistics pass (15 planes read
            # per case, nothing written) and the map is applied by the stem while it loads the raw planes
            nbytes = B * 15 * side * side * 4
            gbs = nbytes / (nm_fused[0] / 1e3) / 1e9
            fused_norm = {"kernel": "dwi_normalize statistics pass (normalisation applied in the stem's operand load)",
                          "ms_per_launch": nm_fused[0], "algorithmic_bytes_per_launch": nbytes, "achieved": gbs,
                          "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                          "note": "instruction-issue bound, not HBM bound: mean / unbiased std / clipped-output mean of a "
                                  "16 KB plane per CTA iteration; it replaces a 0.10 ms read+write pass by a 0.09 ms read pass"}
            # the stand-alone normaliser (public API DWINormalize.batch, and the C4 path) timed here on the same inputs
            pm_tmp = torch.empty(B * dwi_d.shape[1], device=device)
            pipe.dwi_norm.batch(dwi_d, plane_mean=pm_tmp)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            reps = 5
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
            tot = 0.0
            for _ in range(reps):
                flush.zero_()
                ev[0].record()
                pipe.dwi_norm.batch(dwi_d, plane_mean=pm_tmp)
                ev[1].record()
                torch.cuda.synchronize()
                tot += ev[0].elapsed_time(ev[1])
            del flush
            ms_n = tot / reps
            nbytes = B * (15 + 16) * side * side * 4
            gbs = nbytes / (ms_n / 1e3) / 1e9
            hbm_roofline = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": gbs / peaks["hbm_gbs"], "traffic": None,
                            "kernel": "dwi_normalize stand-alone (DWINormalize.batch; L2 flushed between launches)",
                            "ms_per_launch": ms_n, "algorithmic_bytes_per_launch": nbytes}
        conv_ms = sum(sum(t) for (n, _), t in prof.items() if n == "b200_conv_gemm_ex")
        kernels = sorted(((sum(t), n, k, len(t)) for (n, k), t in prof.items()), reverse=True)[:40]
        nsteps_prof = max(2, min(args.steps, 5))
        if args.workload == "c3":
            flop_case = FLOP_PER_CASE_FULL if args.aux == "full" else FLOP_PER_CASE_LOGITS
        elif args.workload == "c4":
            flop_case = FLOP_C4_FULL if args.aux == "full" else FLOP_C4_LOGITS
        else:
            flop_case = FLOP_RESNET
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": {"c3": WORKLOAD, "c4": WORKLOAD_C4, "resnet": WORKLOAD_RESNET}[args.workload] +
                       (" [hybrid TransformerStage encoders]" if args.hybrid else "") +
                       (f" [predict mode {args.predict_mode}: {dict(tta=4, mc=10, tta_mc=40)[args.predict_mode]} forwards per case]"
                        if args.predict_mode != "normal" else ""),
                       "batch_per_gpu": B, "global_batch": B * world, "aux": args.aux,
                       "weights": "seeded random init (initialize_model) + randomised BN running stats",
                       "l2": "no flush needed: per-step inputs (369 MB at B=1024) and activations (>10 GB) exceed the 126 MB L2",
                       "parallelism": f"case-sharded x{world}, one logit all_gather after the K steps" if world > 1 else "single GPU"},
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps, "api": "FusionPipeline.classify_host (pinned host tensors, "
                    "upload overlapped on a copy stream)",
                    "h2d_gbps_needed": h2d / (ms / args.steps) / 1e6,
                    "numa": {k: v for k, v in numa.items() if k != "previous"}},
            "gpu_launches": launches,
            "hbm_peak_allocated_gb": torch.cuda.max_memory_allocated(device) / 1e9,
            "roofline": roofline,
            "roofline_hbm_kernel": hbm_roofline,
            "fused_normalise": fused_norm,
            "step_model": {"algorithmic_gflop_per_case": flop_case / 1e9,
                           "achieved_tflops_whole_step": value / world * flop_case / 1e12,
                           "frac_of_sustained_peak": value / world * flop_case / 1e12 / peaks["tf_sustained"],
                           "conv_gemm_share_of_step": conv_ms / total_ms if total_ms else None,
                           "top_kernels_ms_per_step": [[round(s / nsteps_prof, 3), n, list(k) if k else None, c // nsteps_prof]
                                                       for s, n, k, c in kernels]},
        }
        if not args.no_cpu_baseline and world == 1:  # reported at N=1 only (the other ranks would sit idle)
            line["cpu_baseline"] = run_cpu_baseline(params, cpu_state, nyul, args.cpu_cases, args.ref_batch)
        else:
            line["cpu_baseline"] = None
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))


if __name__ == "__main__":
    main()
