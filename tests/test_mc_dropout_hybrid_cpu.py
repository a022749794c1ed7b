"""CPU: argument checks of the MC-dropout entries of the hybrid transformer stage (b200_attention_mc, b200_linear_mc),
and the MC-dropout oracle of the transformer stage (off: bitwise the eval oracle; on: a random, different output)."""
import torch

import b200_native as nat
import golden_util as gu
import mc_dropout_oracle as mdo
import parameters_default as pd
from oracle import model_oracle as mo
from oracle import params as op


def test_mc_entries_reject_out_of_range_dropout_without_a_gpu():
    """< 0 before anything is launched (the pointers are never read: any non-NULL value stands for a buffer)."""
    lib, p = nat.lib(), 16
    for bad in (-0.1, 1.0, 1.5, float("nan")):
        assert lib.b200_attention_mc(p, 3 * 512, p, 512, 2, 256, 4, 128, 128 ** -0.5, bad, 1, None) < 0
        assert lib.b200_linear_mc(p, 256, 512, p, 512, None, None, p, 1, 2, 0, p, 1, bad, 1, None) < 0  # fp32 res
        assert lib.b200_linear_mc(p, 256, 512, p, 2048, None, None, None, 0, 0, 1, p, 0, bad, 1, None) < 0  # fc1
    assert lib.b200_linear_mc(p, 256, 512, p, 512, None, None, p, 0, 2, 0, p, 0, 0.1, 1, None) < 0  # bf16 residual
    assert lib.b200_linear_mc(p, 256, 512, p, 512, None, None, p, 0, 2, 0, p, 1, 0.1, 1, None) < 0  # bf16 res, fp32 out
    assert lib.b200_linear_mc(p, 256, 512, p, 512, None, None, p, 1, 1, 1, p, 1, 0.1, 1, None) < 0  # act before res


def _hybrid():
    p = pd.default_parameters()
    for m in ("dwi", "dce"):
        p[f"{m}_model_parameters"]["use_hybrid_transformer"] = True
    sd = op.seeded_state_dict(gu.load_shapes("hybrid")["dwi"], seed=7)
    dwi_raw, _, _, _ = op.synthetic_raw(2, seed=1234, kind="S")
    return p, sd, dwi_raw / dwi_raw.amax(dim=(1, 2, 3), keepdim=True)


def test_oracle_transformer_dropout_off_is_bitwise_the_eval_oracle():
    p, sd, dwi = _hybrid()
    mp = p["dwi_model_parameters"]
    torch.set_num_threads(8)
    with torch.no_grad():
        x = torch.randn(2, mp["channels"][1], 32, 32, generator=torch.Generator().manual_seed(3))
        s = mo.SD(sd).sub("transformer")
        ref = mo.transformer_stage(x, s, mp["transformer_heads"], mp["transformer_patch_size"])
        got = mdo.transformer_stage(x, s, mp["transformer_heads"], mp["transformer_patch_size"], 0.0)
        assert torch.equal(got, ref)
        base = mo.encoder_forward(sd, "dwi", p, dwi)[0]
        off = mdo.encoder_forward(sd, "dwi", p, dwi, mc_dropout=False, transformer_dropout=False)[0]
        assert torch.equal(base, off)
    assert mo.transformer_stage is not None and mo.transformer_stage.__module__ == mo.__name__  # restored


def test_oracle_transformer_dropout_on_changes_the_output():
    """Only the transformer's dropouts (p = 0.1): every pass differs from the eval output and from the others."""
    p, sd, dwi = _hybrid()
    torch.set_num_threads(8)
    torch.manual_seed(11)
    with torch.no_grad():
        base = mo.encoder_forward(sd, "dwi", p, dwi)[1]["raw_feats"][2]
        runs = torch.stack([mdo.encoder_forward(sd, "dwi", p, dwi, mc_dropout=False, transformer_dropout=True)[1]
                            ["raw_feats"][2] for _ in range(3)])
    assert all(not torch.equal(r, base) for r in runs)
    spread = runs.std(0).max().item()
    print(f"oracle f3 pass-to-pass spread with the transformer dropouts: {spread:.3e} (max |f3| {base.abs().max():.3e})")
    assert spread > 0
