"""bf16 floor of the ViT-adapter path at 256 x 256 inputs (CPU, oracle only): the configuration of
tests/test_attention_long_gpu.py::test_vit_adapter_pipeline_at_256_vs_oracle (use_backbone ViT-B/16 encoders on
257 tokens, 16 x 16 maps, seeded weights 11, synthetic inputs 4321).

Runs the fp32 oracle twice - once as is, once with every GEMM-shaped op (Conv2d / Linear with >= 64 input channels)
fed bf16-rounded activations and weights (fp32 accumulation, nothing else changed), as tests/tools/bf16_floor.py does
for the 224 x 224 fixture - and prints max|d| / max|ref| per API output.

    python tests/tools/bf16_floor_vit256.py
"""
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import b200path  # noqa: E401,F401
import model_module as mm
from oracle import backbone_oracle as bo, model_oracle as mo, params as op
from test_attention_long_gpu import _inputs, _vit_parameters

torch.set_num_threads(8)
p, bbs = _vit_parameters(256)
mods = {"dwi": mm.ModelMaskHeadBackbone("dwi", p, bbs["dwi"]), "dce": mm.ModelMaskHeadBackbone("dce", p, bbs["dce"]),
        "fusion": mm.FusionModel(p)}
sds = {k: op.seeded_state_dict(op.shapes_of(m.state_dict()), seed=11) for k, m in mods.items()}
dwi, dce = _inputs(2, 256, 4321)
bf = lambda t: t.bfloat16().float()


class Emu:
    """F stand-in that rounds GEMM operands (activations + weights) to bf16, fp32 accumulate."""
    def __getattr__(self, n): return getattr(F, n)

    def conv2d(self, x, w, b=None, **k):
        if w.shape[1] >= 64: x, w = bf(x), bf(w)
        return F.conv2d(x, w, b, **k)

    def linear(self, x, w, b=None):
        if w.shape[1] >= 64: x, w = bf(x), bf(w)
        return F.linear(x, w, b)


def run(emu):
    mo.F = Emu() if emu else F; bo.F = Emu() if emu else F
    out = {}
    with torch.no_grad():
        for m, x in (("dwi", dwi), ("dce", dce)):
            out[m] = mo.encoder_forward(sds[m], m, p, x)
        out["fusion"] = mo.fusion_forward(sds["fusion"], p, out["dwi"][1]["raw_feats"], out["dce"][1]["raw_feats"],
                                          out["dwi"][2], out["dce"][2])
    return out


a = run(False); b = run(True)
def rel(x, y): return ((x - y).abs().max() / y.abs().max()).item()
for m in ("dwi", "dce"):
    print(m, "logits", rel(b[m][0], a[m][0]), "mask", rel(b[m][2], a[m][2]))
    for k, v in a[m][1].items():
        if isinstance(v, list): print(m, k, [round(rel(q, r), 4) for q, r in zip(b[m][1][k], v)])
        elif v is not None: print(m, k, rel(b[m][1][k], v))
print("fusion logits", rel(b["fusion"][0], a["fusion"][0]), "mask", rel(b["fusion"][1], a["fusion"][1]))
for k, v in a["fusion"][2].items():
    if v is not None: print("fusion", k, rel(b["fusion"][2][k], v))
