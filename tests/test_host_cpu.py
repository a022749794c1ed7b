"""CPU-only checks: the C-ABI library exports what include/b200_fusion.h declares, the Python
mirror keeps the reference's parameter names/shapes, host-side logic, loud failure without CUDA."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import b200path
import golden_util as gu

ROOT = b200path.ROOT


def _header_decls():
    text = open(os.path.join(ROOT, "include", "b200_fusion.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    decls = {}
    for m in re.finditer(r"\bint\s+(b200_\w+)\s*\((.*?)\)\s*;", text, flags=re.S):
        args = m.group(2).strip()
        decls[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    return decls


def test_library_exports_every_declared_symbol():
    import b200_native as nat

    decls = _header_decls()
    assert len(decls) >= 15
    lib = nat.lib()  # loads the .so built by __graft_entry__.build(); no GPU needed to load it
    for name, nargs in decls.items():
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in nat.SIGNATURES, f"{name} has no ctypes signature"
        assert len(nat.SIGNATURES[name]) == nargs, f"{name}: ctypes arity != header arity"
    assert set(nat.SIGNATURES) == set(decls)
    assert lib.b200_abi_version() == nat.ABI_VERSION


def test_ex_entry_points_reject_invalid_arguments_without_a_gpu():
    import b200_native as nat

    lib = nat.lib()
    # negative return = invalid argument, nothing launched (no CUDA call is reached)
    assert lib.b200_conv_gemm_ex(None, 64, None, None, None, None, 0, 0, 0, None, 0, 0, None, 64, None, 0, 0, None, 0,
                                 0.0, None, 1, 32, 32, 64, 64, 1, 1, 1, None) < 0
    assert lib.b200_dwi_normalize(None, None, 5, 4, 16, 1, -3.0, 3.0, None, None) < 0   # planes % C != 0
    assert lib.b200_dwi_normalize(None, None, 0, 4, 16, 1, -3.0, 3.0, None, None) == 0  # empty batch is a no-op
    assert lib.b200_nyul_transform_ex(None, None, 6, 6, 16, 40, None, None, None, None, None, 0, None) < 0  # L too large
    assert lib.b200_stem_ex(None, 1, 64, 8, 8, 2, None, None, None, None, None, 0, None, None, None, 8, 8, None, None, None,
                            None, 0.0, 0.0, None, 0, None) < 0


def test_training_kernels_reject_out_of_range_arguments_without_a_gpu():
    """csrc/train_elem.cu: every documented limit returns < 0 before anything is launched (the pointers are never read:
    any non-NULL value stands for a buffer)."""
    import b200_native as nat

    lib, p = nat.lib(), 16
    assert lib.b200_bn_stats(p, 100, 12, 16, p, p, None) == -1                           # C % 8
    assert lib.b200_bn_stats(p, 100, 2056, 2056, p, p, None) == -1                       # C > 2048
    assert lib.b200_bn_finalize(p, p, 8, 0.0, 1e-5, 0.1, None, None, p, p, None) == -1   # count <= 0
    bn = (p, 8, None, 8, p, p, p, p)
    assert lib.b200_bn_act_fwd(p, 16, None, 16, p, p, p, p, 1, 0.0, 0, 10, 12, p, 16, None) == -1   # C % 8
    assert lib.b200_bn_act_fwd(*bn, 3, 0.0, 0, 10, 8, p, 8, None) == -2                  # act
    assert lib.b200_bn_act_fwd(*bn, 1, 1.0, 0, 10, 8, p, 8, None) == -2                  # drop_p >= 1
    assert lib.b200_bn_act_fwd(p, 1032, None, 8, p, p, p, p, 1, 0.0, 0, 10, 1032, p, 1032, None) == -3  # C > 1024
    assert lib.b200_bn_act_bwd(p, 1032, None, 8, p, p, p, p, 1, 0.0, 0, 10, 1032, p, 1032, 1, p, p, 1032, None, 0, p, p,
                               None) == -3
    assert lib.b200_bn_act_bwd(*bn, 1, 0.0, 0, 10, 8, p, 8, 1, p, None, 8, None, 0, p, p, None) == -5  # pass 2 needs dz
    assert lib.b200_bn_act_bwd(*bn, 1, 0.0, 0, 10, 8, p, 8, 1, None, p, 8, None, 0, p, p, None) == -4  # no scratch
    assert lib.b200_map_dot(p, 2056, None, 0, 2, 10, 2056, p, None) == -1                # C > 2048
    assert lib.b200_map_scale_add(p, 16, p, p, 2, 10, 12, p, 16, 0, None) == -1          # C % 8
    assert lib.b200_map_axpby(p, 16, 1.0, None, 0, 0.0, 10, 12, p, 16, None) == -1
    assert lib.b200_map_sumsq(p, 8, 0, 8, p, None) == -1                                 # R <= 0
    assert lib.b200_se_fwd(p, 2, 64, 0, 49, p, p, p, p, p, p, None) == -1                # M <= 0
    assert lib.b200_se_bwd(p, p, p, p, p, p, 2, 6200, 1, p, p, p, p, None) == -2         # shared memory > 48 KB
    for C, taps, H, W in ((24, 9, 8, 8), (288, 1, 8, 8), (64, 4, 8, 8), (64, 9, 200, 200)):  # convc1_shape_ok
        assert lib.b200_convc1_fwd(p, C, 2, H, W, C, taps, p, p, p, None) == -1
        assert lib.b200_convc1_bwd(p, C, p, 2, H, W, C, taps, p, p, C, 0, p, p, None) == -1
    assert lib.b200_convc1_bwd(p, 2048, p, 2, 250, 200, 2048, 1, p, p, 2048, 0, p, p, None) == -2  # dout + dw > 200 KB
    assert lib.b200_lift_fwd(p, 10, 12, p, p, None) == -1                                # N % 8
    assert lib.b200_lift_bwd(p, p, 10, 136, p, p, p, None) == -1                         # N > 128
    assert lib.b200_modulate_bwd(p, 16, p, 16, p, p, 10, 12, p, 16, p, p, None) == -1    # C % 8
    assert lib.b200_mask_attn_bwd(p, p, 2, 256, 33, p, p, p, p, p, 1e-5, p, p, p, p, p, p, None) == -1  # K > 32
    stem = (p, 2, 3, 16, 16)
    assert lib.b200_stem_bwd(*stem, 2, p, p, 264, p, p, p, None) == -1                   # N > 256
    assert lib.b200_stem_bwd(p, 2, 33, 16, 16, 2, p, p, 64, p, p, p, None) == -1         # C > 32
    assert lib.b200_stem_bwd(p, 2, 3, 15, 16, 2, p, p, 64, p, p, p, None) == -1          # H % stride (as b200_stem_ex)
    assert lib.b200_stem_bwd(p, 2, 3, 16, 17, 2, p, p, 64, p, p, p, None) == -1          # W % stride
    assert lib.b200_stem_bwd(*stem, 0, p, p, 64, p, p, p, None) == -1                    # stride < 1
    assert lib.b200_cls_head_bwd(p, p, p, 2, 64, 17, 1, p, p, p, None) == -1             # K > 16
    assert lib.b200_focal_loss(p, p, 2, 17, 0.1, 2.0, None, 1.0, p, p, None) == -1       # K > 16
    assert lib.b200_dice_loss(p, p, 2, 0, 1.0, 1.0, p, p, None) == -1                    # n <= 0
    assert lib.b200_recon_loss(p, 2, 128, 65, p, 1, None, 0, 256, 130, 1e-3, 1.0, p, p, None) == -1  # h w > 8192
    assert lib.b200_recon_loss(p, 2, 16, 16, p, 1, None, 2, 64, 64, 1e-3, 1.0, p, p, None) == -1    # x2 NULL, C2 > 0
    assert lib.b200_mimic_loss(p, p, 2, 12, 1.0, p, p, None) == -1                       # n % 8
    assert lib.b200_gating_fwd(p, p, 0, 64, 49, None, None, 0, p, p, p, p, None) == -1   # B <= 0
    assert lib.b200_gating_bwd(p, p, p, 2, 64, 128, 0, p, p, p, p, None) == -1           # npix <= 0
    assert lib.b200_fused_pool(p, p, 2, 64, 49, None, None, None, 0, p, None) == -1      # alpha NULL
    mix = (p, p, p, p, 2, 14, 14)
    assert lib.b200_fusion_mix_bwd(*mix, 12, 7, 7, p, p, None, None, None, None, None, None, 0, None) == -1  # C % 8
    assert lib.b200_fusion_mix_bwd(*mix, 512, 7, 7, p, p, None, None, None, None, None, None, 0, None) == -3  # smem
    assert lib.b200_fusion_mix_bwd(*mix, 64, 3, 7, None, None, p, p, p, p, p, p, 1, None) == -4  # dtok, H % Hp
    assert lib.b200_mimic_pairs(p, 3, 49, 64, 1.0, p, p, None) == -1                     # B < 4
    assert lib.b200_up2_bwd(p, 2, 7, 7, 12, p, None) == -1                               # C % 8
    assert lib.b200_row_bcast(p, 1, 1.0, 2, 0, p, None) == -1                            # n <= 0
    assert lib.b200_vec_axpby(p, 1.0, 0.0, 0, p, None) == -1                             # n <= 0


def test_missing_library_fails_loudly(monkeypatch):
    import b200_native as nat

    monkeypatch.setattr(nat, "_lib", None)
    monkeypatch.setattr(nat, "LIB_PATH", "/nonexistent/libb200fusion.so")
    with pytest.raises(nat.B200NativeError):
        nat.lib()


@pytest.mark.parametrize("tag,hybrid", [("cnn", False), ("hybrid", True)])
def test_state_dict_matches_reference_names_and_shapes(tag, hybrid):
    import model_module as mm
    import parameters_default as pd

    p = pd.default_parameters()
    for m in ("dwi", "dce"):
        p[f"{m}_model_parameters"]["use_hybrid_transformer"] = hybrid
    ref = gu.load_shapes(tag)
    mods = {"dwi": mm.ModelMaskHeadBackbone("dwi", p), "dce": mm.ModelMaskHeadBackbone("dce", p),
            "fusion": mm.FusionModel(p)}
    for k, m in mods.items():
        mine = {a: tuple(b.shape) for a, b in m.state_dict().items()}
        assert mine == ref[k]


@pytest.mark.parametrize("tag", ["cnn_mf1", "cnn_mf3", "cnn_r2"])
def test_variant_state_dicts_match_reference(tag):
    import model_module as mm
    from test_oracle_golden import variant_parameters

    p, _, shape_tag = variant_parameters(tag)
    ref = gu.load_shapes(shape_tag)
    for k, m in {"dwi": mm.ModelMaskHeadBackbone("dwi", p), "dce": mm.ModelMaskHeadBackbone("dce", p)}.items():
        assert {a: tuple(b.shape) for a, b in m.state_dict().items()} == ref[k]


def test_vit_state_dict_matches_reference_names_and_shapes():
    """use_backbone encoders: same keys as the reference, including the `_orig_mod` level its
    torch._dynamo.disable(backbone) wrapper introduces (model_module.py:539) - checkpoints load unchanged."""
    import model_module as mm
    from test_oracle_golden import vit_parameters

    p, backbones = vit_parameters()
    ref = gu.load_shapes("vit")
    mods = {"dwi": mm.ModelMaskHeadBackbone("dwi", p, backbones["dwi"]),
            "dce": mm.ModelMaskHeadBackbone("dce", p, backbones["dce"]), "fusion": mm.FusionModel(p)}
    for k, m in mods.items():
        mine = {a: tuple(b.shape) for a, b in m.state_dict().items()}
        assert mine == ref[k]
        assert any(a.startswith("backbone._orig_mod.") for a in mine) == (k != "fusion")


def test_resnet_state_dict_matches_reference_names_and_shapes():
    import model_module as mm
    from test_oracle_golden import resnet_parameters

    p, backbones = resnet_parameters()
    assert p["dce_model_parameters"]["backbone_index_lists"] == [[0], [1], [2, 3]]
    assert p["dce_model_parameters"]["downsample"] == (True, False, False)
    ref = gu.load_shapes("resnet")
    for k in ("dwi", "dce"):
        m = mm.ModelMaskHeadBackbone(k, p, backbones[k])
        assert {a: tuple(b.shape) for a, b in m.state_dict().items()} == ref[k]


def test_no_cpu_fallback():
    import b200_native as nat
    import dataset as ds
    import model_module as mm
    import parameters_default as pd

    p = pd.default_parameters()
    enc = mm.ModelMaskHeadBackbone("dwi", p).eval()
    with pytest.raises(nat.B200NativeError):
        enc(torch.zeros(1, 16, 64, 64))
    enc.train()   # the train-mode forward runs on the training kernels: still no CPU path
    with pytest.raises(nat.B200NativeError):
        enc(torch.zeros(1, 16, 64, 64))
    if not torch.cuda.is_available():
        with pytest.raises(nat.B200NativeError):
            ds.DWINormalize()(torch.zeros(4, 8, 8))
    with pytest.raises(nat.B200NativeError):   # stand-alone sub-module forwards are kernel-backed too
        mm.SEBlock(8).eval()(torch.zeros(1, 8, 4, 4))
    with pytest.raises(NotImplementedError):   # ... and in training mode they are driven through their parent
        mm.SEBlock(8).train()(torch.zeros(1, 8, 4, 4))
    import transformer_model as tm
    with pytest.raises(nat.B200NativeError):  # the transformer sub-modules too: CUDA only
        tm.MLP(64).eval()(torch.zeros(1, 4, 64))
    with pytest.raises(nat.B200NativeError):
        tm.TransformerStage(64, 128, depth=1, heads=2).eval()(torch.zeros(1, 64, 8, 8))
    fm = mm.FusionModel(p).train()
    with pytest.raises(nat.B200NativeError):
        fm([torch.zeros(1, 512, 32, 32)], [torch.zeros(1, 512, 32, 32)], torch.zeros(1, 1, 32, 32), torch.zeros(1, 1, 32, 32))


def test_initialize_model_rules():
    import model_module as mm

    lin, bn = torch.nn.Linear(8, 4), torch.nn.BatchNorm2d(16)
    seq = mm.initialize_model(torch.nn.Sequential(lin, bn), False)
    assert all(not q.requires_grad for q in seq.parameters())
    assert torch.count_nonzero(lin.bias) == 0 and torch.count_nonzero(bn.bias) == 0
    assert abs(bn.weight.mean().item() - 1) < 0.05


def test_packed_weight_cache_is_dropped_by_every_weight_rewriting_entry_point():
    """The packed-weight cache keys on (data_ptr, version); writes through `.data` change neither, so
    initialize_model / load_state_dict / .to() and the public invalidate_packed() drop it explicitly."""
    import model_module as mm
    import parameters_default as pd

    p = pd.default_parameters()
    for m in (mm.ModelMaskHeadBackbone("dce", p), mm.FusionModel(p)):
        for poke in (lambda: mm.initialize_model(m, True), lambda: m.load_state_dict(m.state_dict()),
                     lambda: m.to(torch.float32), m.invalidate_packed):
            m._pack_cache = ("sig", "stale")
            poke()
            assert m._pack_cache is None


def test_bilinear_axis_weights_equal_gap_of_interpolate():
    import model_module as mm

    for n_in, n_out in ((4, 32), (4, 14), (3, 7)):
        w = torch.tensor(mm._bilinear_axis_weights(n_in, n_out))
        for i in range(n_in):
            e = torch.zeros(1, 1, n_in, 1)
            e[0, 0, i, 0] = 1.0
            up = F.interpolate(e, size=(n_out, 1), mode="bilinear", align_corners=False)
            assert abs(up.mean().item() - w[i].item()) < 1e-6


def test_nyul_fit_and_tables_are_numpy_exact():
    import preprocess_helpers as pre
    from oracle import normalize_oracle as no
    from oracle import params as op

    gold = gu.load("normalizers.npz")
    _, dce, _, _ = op.synthetic_raw(12, seed=1234, kind="S")
    nyul = pre.NyulStandardizer()
    assert not nyul.fitted
    with pytest.raises(RuntimeError):
        nyul.transform(dce[0])
    nyul.fit(list(dce[:8]), num_channels=6)
    lm = np.stack([nyul.channel_landmarks[c] for c in range(6)])
    assert np.array_equal(lm, gold["nyul/landmarks"]) and np.array_equal(lm, no.nyul_fit(list(dce[:8]), 6))
    prev, gamma = no.percentile_indices(4096, nyul.landmarks)
    x = np.sort(np.random.default_rng(1).random(4096).astype(np.float32))
    manual = np.where(gamma >= 0.5, x[prev + 1] - (x[prev + 1] - x[prev]) * (1 - gamma),
                      x[prev] + (x[prev + 1] - x[prev]).astype(np.float64) * gamma)
    assert np.allclose(manual, np.percentile(x, nyul.landmarks), rtol=0, atol=1e-9)


def test_nyul_save_load_roundtrip(tmp_path):
    import preprocess_helpers as pre

    a = pre.NyulStandardizer()
    a.fit([torch.rand(6, 8, 8) for _ in range(3)], num_channels=6)
    path = str(tmp_path / "lm.npy")
    a.save(path)
    b = pre.NyulStandardizer()
    b.load(path)
    assert b.fitted and all(np.array_equal(a.channel_landmarks[c], b.channel_landmarks[c]) for c in range(6))


def test_collate_and_fold_split():
    import dataset as ds
    import prepare_fusion_model as pf

    items = [(torch.zeros(16, 4, 4), torch.zeros(6, 4, 4), torch.zeros(1, 2, 2), torch.tensor(i % 4)) for i in range(5)]
    d, c, m, y = pf.custom_double_input_collate_fn(items)
    assert d.shape == (5, 16, 4, 4) and c.shape == (5, 6, 4, 4) and m.shape == (5, 1, 2, 2) and y.tolist() == [0, 1, 2, 3, 0]
    d, c, m, y = pf.custom_double_input_collate_fn([it[:2] + it[3:] for it in items])
    assert m is None
    with pytest.raises(RuntimeError):
        pf.custom_double_input_collate_fn([(torch.zeros(1),)])
    labels = torch.arange(40) % 4
    imgs = torch.arange(40).float().view(40, 1, 1, 1)
    seen = []
    for fold in range(5):
        (tr, va), (ltr, lva) = ds.data_segmentation(imgs, labels, 5, 4, fold)
        assert len(tr) + len(va) == 40 and set(tr.flatten().tolist()).isdisjoint(va.flatten().tolist())
        assert sorted(labels[va.flatten().long()].tolist()) == sorted(lva.long().tolist())
        assert [int((lva == k).sum()) for k in range(4)] == [2, 2, 2, 2]
        seen += va.flatten().tolist()
    assert sorted(seen) == list(range(40))


def test_shard_bounds_cover_every_case_once():
    import sharding

    for n, world in ((1024, 8), (10, 4), (3, 8), (0, 2)):
        spans = [sharding.shard_bounds(n, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1]); import b200path, sharding
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
n = 7
lo, hi = sharding.shard_bounds(n, dist.get_rank(), 2)
full = torch.arange(n * 4, dtype=torch.float32).view(n, 4)
got = sharding.gather_logits(full[lo:hi].clone(), n)
assert torch.equal(got, full), got
t = sharding.max_over_ranks(1.0 + dist.get_rank(), "cpu")
assert t == 2.0
dist.destroy_process_group()
print("ok")
"""


def test_logit_gather_two_ranks_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 500)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-batch", "2"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "cases/s" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "port"


def test_batch_augment_draws_torchvision_parameters():
    """dataset.BatchAugment samples what the reference's Compose (RandomAffine -> HFlip -> VFlip,
    code/prepare_single_model.py:107-113) would draw for the same images under the same seed, and restates
    torchvision's inverse affine matrix exactly."""
    import dataset as ds
    from torchvision import transforms as T
    from torchvision.transforms import functional as TF

    aug = ds.BatchAugment(degrees=90, translate=(0.1, 0.1), shear=(0.1, 0.1))
    torch.manual_seed(11)
    mine = aug.sample_params(6, 64, 48)
    torch.manual_seed(11)
    ra = T.RandomAffine(degrees=90, translate=(0.1, 0.1), shear=(0.1, 0.1))
    for k in range(6):
        angle, tr, sc, sh = ra.get_params(ra.degrees, ra.translate, ra.scale, ra.shear, [48, 64])
        hf, vf = bool(torch.rand(1) < 0.5), bool(torch.rand(1) < 0.5)
        assert mine[k] == (angle, tr, sc, sh, hf, vf)
        want = TF._get_inverse_affine_matrix([0.0, 0.0], angle, [float(t) for t in tr], sc, list(sh))
        assert aug.inverse_matrix(angle, tr, sc, sh) == want
    assert aug.inverse_matrix(0.0, (0, 0), 1.0, (0.0, 0.0)) == [1.0, 0.0, 0.0, 0.0, 1.0, 0.0]
    import b200_native as nat
    with pytest.raises(nat.B200NativeError):
        aug.batch(torch.zeros(2, 3, 8, 8))  # CPU tensor: no CPU path
    assert nat.lib().b200_augment(None, None, 0, 3, 8, 8, None, None, 0.0, None) == 0
    assert nat.lib().b200_augment(None, None, 2, 3, 8, 8, None, None, 0.0, None) < 0


def test_reference_checkpoint_layouts_roundtrip(tmp_path):
    """The reference's two on-disk layouts (run_training.py:316-326 dictionary file, Lightning .ckpt state dicts) load
    into the B200 modules: same parameter names and shapes."""
    import checkpoints as ck
    import model_module as mm
    import parameters_default as pd
    from oracle import params as op

    params = pd.default_parameters()
    mods = {"dwi": mm.ModelMaskHeadBackbone("dwi", params), "dce": mm.ModelMaskHeadBackbone("dce", params),
            "fusion": mm.FusionModel(params)}
    want = {}
    for i, (k, m) in enumerate(mods.items()):
        want[k] = op.seeded_state_dict(op.shapes_of(m.state_dict()), seed=20 + i)
        m.load_state_dict(want[k])
    path = str(tmp_path / "fusion_model_dict.pth")
    ck.save_model_dict(path, 0, mods["dwi"], mods["dce"], mods["fusion"])
    ck.save_model_dict(path, 1, mods["dwi"], mods["dce"], mods["fusion"])      # merges, like the reference
    assert sorted(torch.load(path)) == ["dce_0", "dce_1", "dwi_0", "dwi_1", "fusion_0", "fusion_1"]
    fresh = {"dwi": mm.ModelMaskHeadBackbone("dwi", params), "dce": mm.ModelMaskHeadBackbone("dce", params),
             "fusion": mm.FusionModel(params)}
    report = ck.apply_states(ck.load_model_dict(path, 1), **fresh)
    assert all(r == ([], []) for r in report.values())
    for k in fresh:
        got = fresh[k].state_dict()
        assert all(torch.equal(got[n], want[k][n]) for n in want[k])
    with pytest.raises(KeyError):
        ck.load_model_dict(path, 7)
    # Lightning checkpoint of the fusion module: prefixed parameters + foreign entries (metrics) that are dropped
    sd = {}
    for k, prefix in (("dwi", "dwi_model."), ("dce", "dce_model."), ("fusion", "fusion_model.")):
        sd.update({prefix + n: t for n, t in want[k].items()})
    sd["train_acc.mean_value"] = torch.zeros(())
    ckpt = str(tmp_path / "best-v0.ckpt")
    torch.save({"state_dict": sd, "epoch": 3}, ckpt)
    states = ck.load_lightning_checkpoint(ckpt)
    assert sorted(states) == ["dce", "dwi", "fusion"] and set(states["fusion"]) == set(want["fusion"])
    # ... and of a single-modality module (prefix `model.`, prepare_single_model.py:215)
    torch.save({"state_dict": {"model." + n: t for n, t in want["dwi"].items()}}, ckpt)
    single = ck.load_lightning_checkpoint(ckpt)
    assert list(single) == ["model"]
    assert ck.apply_states(single, model=mm.ModelMaskHeadBackbone("dwi", params))["model"] == ([], [])
    with pytest.raises(ValueError):
        ck.split_lightning_state_dict({"foo.bar": torch.zeros(1)})


@pytest.mark.parametrize("name", ["r1_bench_c3.json", "r1_bench_c5.json", "r1_bench_c4.json"])
def test_committed_bench_lines_keep_the_driver_contract(name):
    """The JSON lines bench.py printed on the B200 boxes (profiles/) carry every key of the bench contract."""
    with open(os.path.join(ROOT, "profiles", name)) as f:
        line = json.loads(f.read().strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["unit"] == "cases/s" and line["higher_is_better"] is True and line["scaling"] == "weak"
    assert line["vs_baseline"] is None and line["data"] == "synthetic" and "workload" in line["config"]
    assert line["value"] > 0 and line["gpu_launches"] > 0 and line["warmup"] >= 3
    e2e = line["e2e"]
    assert e2e["value"] > 0 and e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0
    assert e2e["value"] <= 1.02 * line["value"]            # host copies inside the timed region never make it faster
    roof = line["roofline"]
    assert roof["bound"] in ("hbm", "tensor") and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    assert 0.0 < roof["frac"] < 1.0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"])
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(line["clocks"]["reasons"])
    cpu = line["cpu_baseline"]
    assert cpu is None or ({"value", "unit", "cores", "kind", "sample"} <= set(cpu) and cpu["kind"] in ("port", "reference"))


def test_resize_dispatches_the_antialiased_kernel_only_when_a_side_shrinks(monkeypatch):
    """Host logic of dataset.Resize (reference: transforms.Resize(input_size), code/prepare_single_model.py:112-120):
    torchvision antialiases tensors, which differs from plain bilinear taps only where a side shrinks - that, and only
    that, goes to b200_resize_aa_c1; the same size is a no-op; shapes follow (size, size) / (h, w)."""
    import dataset as ds

    calls = []
    monkeypatch.setattr(ds.nat, "resize_aa_c1", lambda src, out: calls.append(("aa", tuple(src.shape), tuple(out.shape))))
    monkeypatch.setattr(ds.nat, "resize_bilinear_c1",
                        lambda src, out: calls.append(("bilinear", tuple(src.shape), tuple(out.shape))))
    x = torch.zeros(2, 3, 64, 64)
    assert ds.Resize(64).batch(x) is x and calls == []
    assert ds.Resize(224).batch(x).shape == (2, 3, 224, 224)
    assert ds.Resize(32).batch(x).shape == (2, 3, 32, 32)
    assert ds.Resize((48, 100)).batch(x).shape == (2, 3, 48, 100)      # one side shrinks, one grows
    assert ds.Resize((64, 100)).batch(x).shape == (2, 3, 64, 100)      # nothing shrinks
    assert calls == [("bilinear", (6, 64, 64), (6, 224, 224)), ("aa", (6, 64, 64), (6, 32, 32)),
                     ("aa", (6, 64, 64), (6, 48, 100)), ("bilinear", (6, 64, 64), (6, 64, 100))]
    with pytest.raises(ValueError):
        ds.Resize(32).batch(torch.zeros(3, 64, 64))
