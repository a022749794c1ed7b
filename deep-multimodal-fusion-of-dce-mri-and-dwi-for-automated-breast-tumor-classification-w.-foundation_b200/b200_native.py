"""ctypes binding of libb200fusion.so - the C ABI declared in include/b200_fusion.h.

This is the only place the Python host layer touches native code.  There is no CPU
fallback: if the shared library is missing, or a tensor is not on a CUDA device, the
call raises.  PyTorch is used for device memory and streams only; every arithmetic
operation of the hot path runs in the hand-written sm_100a kernels.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# csrc/build.sh links the library at <repo>/lib/libb200fusion.so: a short path without the dots and dashes of the
# package directory name, which is the path string dlopen sees.
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libb200fusion.so")
ABI_VERSION = 24

_lib = None


class B200NativeError(RuntimeError):
    pass


class FusionWeights(C.Structure):
    """Mirror of `struct b200_fusion_weights` (include/b200_fusion.h)."""

    _fields_ = [
        ("C", C.c_int), ("T", C.c_int), ("heads", C.c_int), ("se_mid", C.c_int), ("num_classes", C.c_int),
        ("use_cross_attention", C.c_int), ("use_mask_attention", C.c_int), ("use_se", C.c_int),
        ("ln_eps", C.c_float),
        ("gate_w", C.c_void_p), ("gate_b", C.c_void_p),
        ("in_proj_wt", C.c_void_p), ("in_proj_b", C.c_void_p),
        ("out_proj_wt", C.c_void_p), ("out_proj_b", C.c_void_p),
        ("ln_w", C.c_void_p), ("ln_b", C.c_void_p),
        ("ffn1_wt", C.c_void_p), ("ffn1_b", C.c_void_p),
        ("ffn2_wt", C.c_void_p), ("ffn2_b", C.c_void_p),
        ("up_coef", C.c_void_p),
        ("se_w1t", C.c_void_p), ("se_b1", C.c_void_p), ("se_w2t", C.c_void_p), ("se_b2", C.c_void_p),
        ("cls_w", C.c_void_p), ("cls_b", C.c_void_p),
    ]


class GemmDesc(C.Structure):
    """Mirror of `struct b200_gemm_desc` (include/b200_fusion.h)."""

    _fields_ = [
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("heads", C.c_int), ("batch", C.c_int),
        ("a", C.c_void_p), ("a_row_stride", C.c_longlong), ("a_head_stride", C.c_longlong),
        ("a_batch_stride", C.c_longlong), ("a_shared", C.c_int),
        ("b", C.c_void_p), ("b_row_stride", C.c_longlong), ("b_head_stride", C.c_longlong),
        ("b_batch_stride", C.c_longlong),
        ("out", C.c_void_p), ("out_row_stride", C.c_longlong), ("out_head_stride", C.c_longlong),
        ("out_batch_stride", C.c_longlong),
        ("res", C.c_void_p), ("res_row_stride", C.c_longlong), ("res_head_stride", C.c_longlong),
        ("res_batch_stride", C.c_longlong),
        ("res_mode", C.c_int), ("act", C.c_int),
        ("scale", C.c_void_p), ("bias", C.c_void_p), ("vec_h_stride", C.c_int),
        ("rowscale", C.c_void_p), ("mode", C.c_int), ("alpha", C.c_float), ("n_valid", C.c_int),
        ("rowsum_inv", C.c_void_p), ("b_rows", C.c_int),
    ]


class HeadTrain(C.Structure):
    """Mirror of `struct b200_head_train` (include/b200_fusion.h)."""

    _fields_ = [
        ("C", C.c_int), ("T", C.c_int), ("se_mid", C.c_int), ("num_classes", C.c_int),
        ("use_mask_attention", C.c_int), ("use_se", C.c_int), ("npix_mask", C.c_int),
        ("smoothing", C.c_float), ("gamma", C.c_float), ("loss_scale", C.c_float),
        ("class_weights", C.c_void_p), ("tok_dwi", C.c_void_p), ("tok_dce", C.c_void_p), ("lowres", C.c_void_p),
        ("mask_dwi", C.c_void_p), ("mask_dce", C.c_void_p), ("labels", C.c_void_p),
        ("gate_w", C.c_void_p), ("gate_b", C.c_void_p), ("up_coef", C.c_void_p),
        ("se_w1", C.c_void_p), ("se_b1", C.c_void_p), ("se_w2", C.c_void_p), ("se_b2", C.c_void_p),
        ("cls_w", C.c_void_p), ("cls_b", C.c_void_p),
        ("loss_out", C.c_void_p), ("logits_out", C.c_void_p), ("gating_out", C.c_void_p),
        ("dlogits_out", C.c_void_p), ("z_out", C.c_void_p), ("gf_out", C.c_void_p), ("h_out", C.c_void_p),
        ("da1_out", C.c_void_p), ("da2_out", C.c_void_p), ("gx_out", C.c_void_p), ("dgl_out", C.c_void_p),
        ("dpd_out", C.c_void_p), ("dpc_out", C.c_void_p), ("dlowres_out", C.c_void_p),
        ("forward_only", C.c_int), ("mask_v", C.c_void_p), ("mk_tmpd", C.c_void_p), ("mk_tmpc", C.c_void_p),
        ("mk_q", C.c_void_p), ("gate_out", C.c_void_p), ("u_out", C.c_void_p), ("dug_out", C.c_void_p),
        ("aud_out", C.c_void_p), ("auc_out", C.c_void_p),
        ("pvec_dwi", C.c_void_p), ("pvec_dce", C.c_void_p), ("pvec_scale", C.c_float),
    ]


_P, _I, _F, _LL = C.c_void_p, C.c_int, C.c_float, C.c_longlong

# name -> argtypes; must list every symbol include/b200_fusion.h declares (tests check this).
SIGNATURES = {
    "b200_abi_version": [],
    "b200_conv_gemm_ex": [_P, _I, _P, _P, _P, _P, _I, _I, _I, _P, _I, _I, _P, _I, _P, _I, _I, _P, _I, _F, _P, _I, _I, _I,
                          _I, _I, _I, _I, _I, _P],
    "b200_conv_gemm_mc": [_P, _I, _P, _P, _P, _P, _I, _I, _I, _P, _I, _I, _P, _I, _P, _I, _I, _P, _I, _F, _P, _I, _I, _I,
                          _I, _I, _I, _I, _I, _F, C.c_ulonglong, _I, _P],
    "b200_attention": [_P, _I, _P, _I, _I, _I, _I, _I, _F, _P],
    "b200_attention_mc": [_P, _I, _P, _I, _I, _I, _I, _I, _F, _F, C.c_ulonglong, _P],
    "b200_resize_bilinear_c1": [_P, _I, _I, _I, _P, _I, _I, _P],
    "b200_resize_aa_c1": [_P, _I, _I, _I, _P, _I, _I, _P],
    "b200_mask_attention": [_P, _I, _I, _I, _P, _P, _P, _P, _P, _F, _P, _P],
    "b200_tapsum": [_P, _I, _I, _I, _P, _P, _P],
    "b200_gemm_batched": [C.POINTER(GemmDesc), _P],
    "b200_layernorm": [_P, _I, _LL, _I, _P, _P, _F, _P, _I, _P],
    "b200_patchify": [_P, _P, _I, _I, _I, _I, _I, _P, _P],
    "b200_vit_tokens": [_P, _P, _P, _I, _I, _I, _P, _P],
    "b200_vit_feature": [_P, _I, _I, _I, _P, _I, _P],
    "b200_linear": [_P, _LL, _I, _P, _I, _P, _P, _P, _I, _I, _I, _P, _I, _P],
    "b200_linear_mc": [_P, _LL, _I, _P, _I, _P, _P, _P, _I, _I, _I, _P, _I, _F, C.c_ulonglong, _P],
    "b200_dwi_normalize": [_P, _P, _I, _I, _I, _I, _F, _F, _P, _P],
    "b200_dwi_normalize_ex": [_P, _P, _I, _I, _I, _I, _F, _F, _P, _P, _P],
    "b200_nyul_transform_ex2": [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P],
    "b200_stem_ex": [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, _P, _F, _F, _P, _I, _P],
    "b200_stem_mc": [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, _P, _F, _F, _P, _I, _F,
                     C.c_ulonglong, _P],
    "b200_nyul_transform_ex": [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P],
    "b200_plane_mean": [_P, _I, _I, _P, _P],
    "b200_case_max_scale": [_P, _I, _LL, _P, _P],
    "b200_se_gate": [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P],
    "b200_scale_map": [_P, _P, _I, _I, _I, _P, _P, _P, _P],
    "b200_conv3x3_c1": [_P, _I, _I, _I, _I, _P, _P, _P, _P],
    "b200_mask_tail": [_P, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _F, _P, _P],
    "b200_lift_c1": [_P, _LL, _I, _P, _P, _P, _P, _P],
    "b200_cls_head": [_P, _P, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P],
    "b200_channel_sums": [_P, _I, _I, _I, _I, _P, _P],
    "b200_mix_instnorm": [_P, _P, _I, _I, _I, _P, _P, _P, _F, _P, _P],
    "b200_adaptive_pool": [_P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "b200_add_maps": [_P, _P, _LL, _P, _P],
    "b200_adc_map": [_P, _I, _I, _I, _P, _F, _P, _P],
    "b200_maxpool3x3_s2": [_P, _I, _I, _I, _I, _P, _P],
    "b200_im2col7x7_s2": [_P, _P, _I, _I, _I, _I, _I, _P, _P],
    "b200_flip_planes": [_P, _P, _LL, _I, _I, _I, _I, _P],
    "b200_augment": [_P, _P, _I, _I, _I, _I, _P, _P, _F, _P],
    "b200_fusion_tokens": [_P, _I, _I, _I, _I, _I, _I, _P, _P],
    "b200_fusion_core": [C.POINTER(FusionWeights), _I, _P, _P, _I, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P],
    "b200_fusion_mix": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P],
    "b200_sgemm": [_P, _LL, _I, _P, _LL, _I, _P, _LL, _I, _I, _I, _P, _P, _LL, _I, _P, _I, _I, _I, _P],
    "b200_colsum": [_P, _LL, _I, _I, _P, _P],
    "b200_mha_fwd": [_P, _LL, _P, _P, _LL, _I, _I, _I, _I, _I, _P, _P, _LL, _P],
    "b200_mha_bwd": [_P, _LL, _P, _P, _LL, _P, _P, _LL, _I, _I, _I, _I, _I, _P, _P, _P, _P],
    "b200_ln_fwd": [_P, _I, _I, _P, _P, _F, _P, _P, _P, _P],
    "b200_ln_bwd": [_P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P],
    "b200_gelu_bwd": [_P, _P, _LL, _P, _P],
    "b200_head_loss": [C.POINTER(HeadTrain), _I, _P],
    "b200_adamw": [_P, _P, _P, _P, _LL, _F, _F, _F, _F, _F, _I, _F, _P],
    "b200_adamw_groups": [_P, _P, _P, _P, _LL, _P, _P, _P, _F, _F, _F, _F, _I, _F, _P],
    "b200_mask_dot": [_P, _P, _I, _I, _I, _P, _P],
    "b200_mask_dice": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _F, _F, _I, _P,
                       _P, _P, _P, _P, _P],
    "b200_mask_wsum": [_P, _P, _I, _I, _I, _P, _P],
    "b200_mask_head_grads": [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P],
    "b200_conv_wgrad": [_P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, _P],
    "b200_pack_conv_weights": [_P, _I, _I, _I, _P, _P, _P],
    "b200_bn_stats": [_P, _LL, _I, _I, _P, _P, _P],
    "b200_bn_finalize": [_P, _P, _I, C.c_double, _F, _F, _P, _P, _P, _P, _P],
    "b200_bn_act_fwd": [_P, _I, _P, _I, _P, _P, _P, _P, _I, _F, C.c_ulonglong, _LL, _I, _P, _I, _P],
    "b200_bn_act_bwd": [_P, _I, _P, _I, _P, _P, _P, _P, _I, _F, C.c_ulonglong, _LL, _I, _P, _I, _I, _P, _P, _I, _P, _I,
                        _P, _P, _P],
    "b200_map_dot": [_P, _I, _P, _I, _I, _I, _I, _P, _P],
    "b200_map_scale_add": [_P, _I, _P, _P, _I, _I, _I, _P, _I, _I, _P],
    "b200_map_axpby": [_P, _I, _F, _P, _I, _F, _LL, _I, _P, _I, _P],
    "b200_map_sumsq": [_P, _I, _LL, _I, _P, _P],
    "b200_se_fwd": [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P],
    "b200_se_bwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P],
    "b200_convc1_fwd": [_P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P],
    "b200_convc1_bwd": [_P, _I, _P, _I, _I, _I, _I, _I, _P, _P, _I, _I, _P, _P, _P],
    "b200_lift_fwd": [_P, _LL, _I, _P, _P, _P],
    "b200_lift_bwd": [_P, _P, _LL, _I, _P, _P, _P, _P],
    "b200_modulate_bwd": [_P, _I, _P, _I, _P, _P, _LL, _I, _P, _I, _P, _P, _P],
    "b200_mask_attn_bwd": [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _F, _P, _P, _P, _P, _P, _P, _P],
    "b200_stem_bwd": [_P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P, _P, _P],
    "b200_cls_head_bwd": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P],
    "b200_focal_loss": [_P, _P, _I, _I, _F, _F, _P, _F, _P, _P, _P],
    "b200_dice_loss": [_P, _P, _I, _I, _F, _F, _P, _P, _P],
    "b200_recon_loss": [_P, _I, _I, _I, _P, _I, _P, _I, _I, _I, _F, _F, _P, _P, _P],
    "b200_gating_fwd": [_P, _P, _I, _I, _I, _P, _P, _I, _P, _P, _P, _P, _P],
    "b200_gating_bwd": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P],
    "b200_fused_pool": [_P, _P, _I, _I, _I, _P, _P, _P, _I, _P, _P],
    "b200_fusion_mix_bwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P],
    "b200_mimic_pairs": [_P, _I, _I, _I, _F, _P, _P, _P],
    "b200_mimic_loss": [_P, _P, _I, _LL, _F, _P, _P, _P],
    "b200_up2_bwd": [_P, _I, _I, _I, _I, _P, _P],
    "b200_vec_axpby": [_P, _F, _F, _LL, _P, _P],
    "b200_row_bcast": [_P, _I, _F, _I, _I, _P, _P],
}


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200NativeError(
                f"{LIB_PATH} is missing: build it with csrc/build.sh (or __graft_entry__.build()); "
                "this package has no CPU or PyTorch fallback")
        path = LIB_PATH
        # a checkout reached through the /root/repo symlink is opened under that name (same file, plain path)
        alias = "/root/repo/lib/libb200fusion.so"
        if path != alias and os.path.exists(alias) and os.path.samefile(alias, path):
            path = alias
        handle = C.CDLL(path)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = C.c_int
        if handle.b200_abi_version() != ABI_VERSION:
            raise B200NativeError("libb200fusion.so ABI version mismatch; rebuild it")
        _lib = handle
    return _lib


def _ptr(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise B200NativeError("b200 native ops need CUDA tensors (there is no CPU path)")
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check(rc, name):
    if rc != 0:
        kind = "invalid argument" if rc < 0 else "CUDA error"
        raise B200NativeError(f"{name} failed: {kind} {rc}")


LAUNCH_COUNT = 0   # kernels launched through this binding (bench.py reports it as gpu_launches)
_profile = None    # list of (name, key, start_event, end_event) while profiling


def start_profile():
    """Bracket every subsequent native launch with CUDA events on the launching stream."""
    global _profile
    _profile = []


def stop_profile():
    """-> {(name, key): [ms, ...]} for the launches since start_profile() (synchronises)."""
    global _profile
    rec, _profile = _profile, None
    torch.cuda.synchronize()
    out = {}
    for name, key, s, e in rec or []:
        out.setdefault((name, key), []).append(s.elapsed_time(e))
    return out


def _call(name, key, *args):
    global LAUNCH_COUNT
    fn = getattr(lib(), name)
    if _profile is not None:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rc = fn(*args)
        e.record()
        _profile.append((name, key, s, e))
    else:
        rc = fn(*args)
    LAUNCH_COUNT += 1
    _check(rc, name)


def _bf16_map(t, name, allow_slice=False):
    """NHWC bf16 map; with allow_slice also a channel slice [..., a:b] of a contiguous NHWC buffer (its row stride
    is then the wider buffer's channel count)."""
    if t.dtype != torch.bfloat16:
        raise B200NativeError(f"{name} must be a bfloat16 NHWC tensor")
    if t.is_contiguous():
        return
    B, H, W, _ = t.shape
    ld = t.stride(2)
    if not (allow_slice and t.stride(3) == 1 and t.stride(1) == W * ld and t.stride(0) == H * W * ld and ld % 8 == 0):
        raise B200NativeError(f"{name} must be a contiguous bfloat16 NHWC tensor (or a channel slice of one)")


def _ld(t):
    return t.stride(2) if t.dim() == 4 else t.shape[-1]


def conv_gemm(x, w, *, taps, scale=None, bias=None, res=None, res_mode=0, act=0, out=None, up2=False, gap=None,
              cin=None, store=True, n_split=None, act2=0, out2=None, dot_w=None, dot_out=None, dot_bias=0.0, stride=1,
              dropout=None, dilation=1):
    """x [B,H,W,ld] bf16 NHWC (channels [0,cin) used); w [Cout, taps*cin] bf16.  Returns `out`
    (or (out, out2) when n_split is given: channels [n_split, Cout) form a second layer on the same input)."""
    _bf16_map(x, "x", allow_slice=True)
    B, H, W, _ = x.shape
    x_ld = _ld(x)
    cin = x.shape[-1] if cin is None else cin
    cout = w.shape[0]
    assert w.dtype == torch.bfloat16 and w.is_contiguous() and w.shape[1] == taps * cin
    n1 = cout if n_split is None else n_split
    cs = 2 if taps == 4 else stride
    if out is None and store:
        oh, ow = (2 * H, 2 * W) if up2 else (H // cs, W // cs)
        out = torch.empty((B, oh, ow, n1), dtype=torch.bfloat16, device=x.device)
    if n_split is not None and out2 is None:
        out2 = torch.empty((B, H // cs, W // cs, cout - n_split), dtype=torch.bfloat16, device=x.device)
    if gap is not None and taps == 4:
        raise B200NativeError("gap with the strided patch-embedding conv is not supported")
    out_ld = _ld(out) if out is not None else 0
    if out is not None:
        _bf16_map(out, "out", allow_slice=True)
    if out2 is not None:
        _bf16_map(out2, "out2", allow_slice=True)
    if res is not None:
        _bf16_map(res, "res")
    key = (B, H, W, cin, cout, taps) if stride == 1 else (B, H, W, cin, cout, taps, stride)
    args = (_ptr(x), x_ld, _ptr(w), _ptr(scale), _ptr(bias), _ptr(res), res.shape[-1] if res is not None else 0,
            res_mode, act, _ptr(out), out_ld, 1 if up2 else 0, _ptr(gap), n1, _ptr(out2),
            _ld(out2) if out2 is not None else 0, act2, _ptr(dot_w), dot_w.shape[0] if dot_w is not None else 0,
            float(dot_bias), _ptr(dot_out), B, H, W, cin, cout, taps, stride, dilation)
    if dropout is not None:  # (p, seed, segments): the MC-dropout epilogue, part of this launch's argument list
        p_drop, seed, segments = dropout
        _call("b200_conv_gemm_mc", key, *args, float(p_drop), int(seed) & 0xFFFFFFFFFFFFFFFF, int(segments), _stream())
    else:
        _call("b200_conv_gemm_ex", key, *args, _stream())
    return out if n_split is None else (out, out2)


def gemm_batched(*, M, N, K, heads, batch, a, a_strides, b, b_strides, out, out_strides, a_shared=False, res=None,
                 res_strides=(0, 0, 0), res_mode=0, act=0, scale=None, bias=None, vec_h_stride=0, rowscale=None,
                 mode=0, alpha=1.0, n_valid=0, rowsum_inv=None, b_rows=0):
    """Batched K-major GEMM (see b200_gemm_batched).  a / b / out / res are data pointers (ints) so that views
    with channel offsets can be passed; strides are (row, head, batch) in elements."""
    d = GemmDesc()
    d.M, d.N, d.K, d.heads, d.batch = M, N, K, heads, batch
    d.a, (d.a_row_stride, d.a_head_stride, d.a_batch_stride), d.a_shared = a, a_strides, int(a_shared)
    d.b, (d.b_row_stride, d.b_head_stride, d.b_batch_stride) = b, b_strides
    d.out, (d.out_row_stride, d.out_head_stride, d.out_batch_stride) = out, out_strides
    d.res, (d.res_row_stride, d.res_head_stride, d.res_batch_stride) = res, res_strides
    d.res_mode, d.act = res_mode, act
    d.scale, d.bias, d.vec_h_stride = _ptr(scale), _ptr(bias), vec_h_stride
    d.rowscale, d.mode, d.alpha, d.n_valid, d.rowsum_inv = _ptr(rowscale), mode, float(alpha), n_valid, _ptr(rowsum_inv)
    d.b_rows = b_rows
    _call("b200_gemm_batched", (batch, heads, M, K, N, mode), C.byref(d), _stream())


def layernorm(x, w, b, eps, out=None, out_dtype=torch.bfloat16):
    """x [rows, C] bf16 or fp32 contiguous -> LayerNorm over C, bf16 (default) or fp32."""
    rows, C_ = x.numel() // x.shape[-1], x.shape[-1]
    if out is None:
        out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    _call("b200_layernorm", None, _ptr(x), int(x.dtype == torch.float32), rows, C_, _ptr(w), _ptr(b), float(eps),
          _ptr(out), int(out.dtype == torch.float32), _stream())
    return out


def linear_f32(x2d, w, *, scale=None, bias=None, res=None, res_mode=0, act=0, out=None, out_dtype=torch.bfloat16,
               dropout=None):
    """x2d [M,K] bf16, w [N,K] bf16; residual / output may be fp32 [M,N] (the transformer residual stream).
    dropout = (p, seed): MC dropout before the residual add, out = res + drop(act(x w^T * scale + bias))
    (b200_linear_mc)."""
    M, K = x2d.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=x2d.device)
    args = (_ptr(x2d), M, K, _ptr(w), N, _ptr(scale), _ptr(bias), _ptr(res),
            int(res is not None and res.dtype == torch.float32), res_mode, act, _ptr(out), int(out.dtype == torch.float32))
    if dropout is not None:
        _call("b200_linear_mc", (M, K, N), *args, float(dropout[0]), int(dropout[1]) & 0xFFFFFFFFFFFFFFFF, _stream())
    else:
        _call("b200_linear", (M, K, N), *args, _stream())
    return out


def patchify(x, P, out, gate=None):
    """`gate` [B,C] fp32 (optional) multiplies plane (b, c) on the way in (modality attention)."""
    B, C_, H, W = x.shape
    _call("b200_patchify", None, _ptr(x), _ptr(gate), B, C_, H, W, P, _ptr(out), _stream())
    return out


def vit_tokens(patches, cls, pos, B, n_patch, E, t):
    _call("b200_vit_tokens", None, _ptr(patches), _ptr(cls), _ptr(pos), B, n_patch, E, _ptr(t), _stream())
    return t


def vit_feature(t, B, n_patch, E, out, out_ld=None):
    """`out` may be a channel slice of a wider [B, n, out_ld] buffer (pass its row stride as out_ld)."""
    _call("b200_vit_feature", None, _ptr(t), B, n_patch, E, _ptr(out), E if out_ld is None else out_ld, _stream())
    return out


def channel_sums(x, out=None):
    """x [B,H,W,C] bf16 NHWC (the last dim may be a channel slice of a wider row) -> [B,C] fp32 sums."""
    B, H, W, C_ = x.shape
    if out is None:
        out = torch.empty((B, C_), dtype=torch.float32, device=x.device)
    _call("b200_channel_sums", None, _ptr(x), x.stride(2), B, H * W, C_, _ptr(out), _stream())
    return out


def mix_instnorm(fb, f, weight_logit, gn_w, gn_b, eps, out=None):
    """GroupNorm(C, C)(sigmoid(w) * fb + (1 - sigmoid(w)) * f) on contiguous NHWC bf16 maps."""
    B, H, W, C_ = f.shape
    if out is None:
        out = torch.empty_like(f)
    _call("b200_mix_instnorm", None, _ptr(fb), _ptr(f), B, H * W, C_, _ptr(weight_logit), _ptr(gn_w), _ptr(gn_b),
          float(eps), _ptr(out), _stream())
    return out


def adaptive_pool(x, size, act=0):
    """x [B,H,W,C] bf16 NHWC -> [B,size,size,C] bf16 (optional GELU), or x [B,H,W] fp32 -> [B,size,size] fp32."""
    if x.dim() == 3:
        B, H, W = x.shape
        out = torch.empty((B, size, size), dtype=torch.float32, device=x.device)
        _call("b200_adaptive_pool", None, _ptr(x), 1, B, H, W, 1, size, size, 0, _ptr(out), _stream())
        return out
    B, H, W, C_ = x.shape
    out = torch.empty((B, size, size, C_), dtype=torch.bfloat16, device=x.device)
    _call("b200_adaptive_pool", None, _ptr(x), 0, B, H, W, C_, size, size, act, _ptr(out), _stream())
    return out


def add_maps(a, b, out=None):
    if out is None:
        out = torch.empty_like(a)
    _call("b200_add_maps", None, _ptr(a), _ptr(b), a.numel(), _ptr(out), _stream())
    return out


def tapsum(d, bias, out):
    B, H, W, _ = d.shape
    _call("b200_tapsum", None, _ptr(d), B, H, W, _ptr(bias), _ptr(out), _stream())
    return out


def linear(x2d, w, *, scale=None, bias=None, res=None, res_mode=0, act=0, out=None, dropout=None):
    """Plain GEMM: x2d [M,K] bf16, w [N,K] bf16 -> [M,N] bf16 with the same fused epilogue.  dropout = (p, seed): MC
    dropout after the activation (and after a residual), element (row, col) decided by Philox(seed; row * N + col)."""
    M, K = x2d.shape
    y = conv_gemm(x2d.view(1, 1, M, K), w, taps=1, scale=scale, bias=bias,
                  res=None if res is None else res.view(1, 1, M, -1), res_mode=res_mode, act=act,
                  out=None if out is None else out.view(1, 1, M, -1),
                  dropout=None if dropout is None else (dropout[0], dropout[1], 1))
    return y.view(M, -1)


def dwi_normalize(x, out, C_, n, skip_last, z_lo, z_hi, plane_mean=None):
    planes = x.numel() // n
    _call("b200_dwi_normalize", None, _ptr(x), _ptr(out), planes, C_, n, 1 if skip_last else 0, float(z_lo),
                                    float(z_hi), _ptr(plane_mean), _stream())
    return out


def nyul_transform(x, out, C_, n, avg_landmarks, standard_scale, prev_index, gamma, plane_mean=None, exact=False):
    """exact=False: composed piece-wise linear table per plane (<= 1 fp32 ulp from numpy); exact=True: numpy's own
    fp64 operation order (bit-identical on > 99.9 % of the samples, ~6x the instructions)."""
    planes = x.numel() // n
    L = standard_scale.numel()
    _call("b200_nyul_transform_ex", None, _ptr(x), _ptr(out), planes, C_, n, L, _ptr(avg_landmarks),
          _ptr(standard_scale), _ptr(prev_index), _ptr(gamma), _ptr(plane_mean), 1 if exact else 0, _stream())
    return out


def attention(qkv, out, B, N, heads, dh, scale=None, dropout=None):
    """Fused softmax(q k^T * scale) v over the packed qkv rows [B*N, 3*heads*dh] bf16 -> out [B*N, heads*dh] bf16
    (b200_attention; transformer_model.py:101-112).  dropout = (p, seed): attention dropout on the probabilities
    (b200_attention_mc)."""
    assert qkv.dtype == torch.bfloat16 and out.dtype == torch.bfloat16 and qkv.stride(-1) == 1 and out.stride(-1) == 1
    args = (_ptr(qkv), qkv.stride(0), _ptr(out), out.stride(0), B, N, heads, dh,
            float(dh ** -0.5 if scale is None else scale))
    if dropout is not None:
        _call("b200_attention_mc", (B, N, heads, dh), *args, float(dropout[0]), int(dropout[1]) & 0xFFFFFFFFFFFFFFFF,
              _stream())
    else:
        _call("b200_attention", (B, N, heads, dh), *args, _stream())
    return out


def plane_mean(x, planes, n, out):
    _call("b200_plane_mean", None, _ptr(x), planes, n, _ptr(out), _stream())
    return out


def adc_map(x, bvals, eps=1e-6):
    """x [B,C,H,W] fp32 CUDA, bvals [C] fp32 CUDA -> [B,1,H,W] ADC maps."""
    x = x.contiguous().float()
    B, C_, H, W = x.shape
    out = torch.empty((B, 1, H, W), dtype=torch.float32, device=x.device)
    _call("b200_adc_map", None, _ptr(x), B, C_, H * W, _ptr(bvals), float(eps), _ptr(out), _stream())
    return out


def im2col7x7_s2(x, gate, kp):
    """x [B,C,H,W] fp32 -> bf16 patch matrix [B*H/2*W/2, kp] of the 7x7 / stride-2 stem."""
    x = x.contiguous().float()
    B, C_, H, W = x.shape
    out = torch.empty((B * (H // 2) * (W // 2), kp), dtype=torch.bfloat16, device=x.device)
    _call("b200_im2col7x7_s2", None, _ptr(x), _ptr(gate), B, C_, H, W, kp, _ptr(out), _stream())
    return out


def maxpool3x3_s2(x):
    B, H, W, C_ = x.shape
    y = torch.empty((B, H // 2, W // 2, C_), dtype=torch.bfloat16, device=x.device)
    _call("b200_maxpool3x3_s2", None, _ptr(x), B, H, W, C_, _ptr(y), _stream())
    return y


def flip_planes(x, flip_w, flip_h):
    """torch.flip over the last / second-last dimension of an fp32 CUDA tensor [..., H, W] (out of place)."""
    x = x.contiguous().float()
    out = torch.empty_like(x)
    H, W = x.shape[-2], x.shape[-1]
    _call("b200_flip_planes", None, _ptr(x), _ptr(out), x.numel() // (H * W), H, W, int(flip_w), int(flip_h), _stream())
    return out


def stem(x, stride, pm, se, wcat, scale, bias, n_skip, n_mid, skip_out, mid_out, mod_attn, dropout=None, input_norm=None):
    """input_norm: None (x is normalised), ("dwi", stats [B*C,4] fp32, z_lo, z_hi) or ("nyul", tables [B*C,56] fp64, L):
    x is the RAW input and the normalisation is applied in the operand load (b200_stem_ex)."""
    B, C_, H, W = x.shape
    w1, b1, w2, b2 = se if se is not None else (None, None, None, None)
    cm = w1.shape[0] if w1 is not None else 0
    aff = tab = None
    z_lo = z_hi = 0.0
    L = 0
    if input_norm is not None:
        if input_norm[0] == "dwi":
            _, aff, z_lo, z_hi = input_norm
        else:
            _, tab, L = input_norm
    args = (_ptr(x), B, C_, H, W, stride, _ptr(pm), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), cm, _ptr(wcat), _ptr(scale),
            _ptr(bias), n_skip, n_mid, _ptr(skip_out), _ptr(mid_out), _ptr(mod_attn), _ptr(aff), float(z_lo), float(z_hi),
            _ptr(tab), int(L))
    if dropout is not None:  # (p, seed): MC dropout on the bottleneck output
        _call("b200_stem_mc", None, *args, float(dropout[0]), int(dropout[1]) & 0xFFFFFFFFFFFFFFFF, _stream())
    else:
        _call("b200_stem_ex", None, *args, _stream())


def se_gate(gap_sum, npix, w1t, b1, w2t, b2, gate):
    B, C_ = gap_sum.shape
    hidden = torch.empty((B, w1t.shape[1]), dtype=torch.float32, device=gap_sum.device)
    _call("b200_se_gate", None, _ptr(gap_sum), B, C_, w1t.shape[1], npix, _ptr(w1t), _ptr(b1), _ptr(w2t), _ptr(b2),
                              _ptr(gate), _ptr(hidden), _stream())
    global LAUNCH_COUNT
    LAUNCH_COUNT += 1  # the call launches two kernels (hidden layer, gate layer)
    return gate


def scale_map(x, y, gate=None, attn=None, gamma=None):
    B, H, W, C_ = x.shape
    _call("b200_scale_map", None, _ptr(x), _ptr(y), B, H * W, C_, _ptr(gate), _ptr(attn), _ptr(gamma), _stream())
    return y


def conv3x3_c1(x, w, bias, out):
    B, H, W, C_ = x.shape
    _call("b200_conv3x3_c1", None, _ptr(x), B, H, W, C_, _ptr(w), _ptr(bias), _ptr(out), _stream())
    return out


def mask_tail(pre, w_out, b_out, mask_pred, attn_params=None, attn=None):
    B, H, W, Cm = pre.shape
    if attn_params is None:
        hc, wa, gw, gb, wb, bb, eps = 0, None, None, None, None, None, 0.0
    else:
        hc, wa, gw, gb, wb, bb, eps = attn_params
    _call("b200_mask_tail", None, _ptr(pre), B, H * W, Cm, _ptr(w_out), _ptr(b_out), _ptr(mask_pred), hc, _ptr(wa),
                                _ptr(gw), _ptr(gb), _ptr(wb), _ptr(bb), float(eps), _ptr(attn), _stream())


def mask_attention(mask, attn_params, attn):
    B = mask.shape[0]
    hc, wa, gw, gb, wb, bb, eps = attn_params
    _call("b200_mask_attention", None, _ptr(mask), B, mask[0].numel(), hc, _ptr(wa), _ptr(gw), _ptr(gb), _ptr(wb),
          _ptr(bb), float(eps), _ptr(attn), _stream())
    return attn


def resize_bilinear_c1(src, out):
    """src [B,h,w] fp32 -> out [B,H,W] fp32, F.interpolate(bilinear, align_corners=False)."""
    B, h, w = src.shape
    _call("b200_resize_bilinear_c1", None, _ptr(src), B, h, w, _ptr(out), out.shape[-2], out.shape[-1], _stream())
    return out


def resize_aa_c1(src, out):
    """src [B,h,w] fp32 -> out [B,H,W] fp32, F.interpolate(bilinear, align_corners=False, antialias=True)."""
    B, h, w = src.shape
    _call("b200_resize_aa_c1", None, _ptr(src), B, h, w, _ptr(out), out.shape[-2], out.shape[-1], _stream())
    return out


def lift_c1(r, w, scale, bias, y):
    _call("b200_lift_c1", None, _ptr(r), r.numel(), w.numel(), _ptr(w), _ptr(scale), _ptr(bias), _ptr(y), _stream())
    return y


def cls_head(gap_sum, gate, npix, fc_w, fc_b, normalize, logits, pooled_out=None):
    B, C_ = gap_sum.shape
    _call("b200_cls_head", None, _ptr(gap_sum), _ptr(gate), B, C_, npix, fc_w.shape[0], _ptr(fc_w), _ptr(fc_b),
                               1 if normalize else 0, _ptr(logits), _ptr(pooled_out), _stream())
    return logits


def fusion_tokens(p, hp, wp, tokens):
    B, H, W, C_ = p.shape
    _call("b200_fusion_tokens", None, _ptr(p), B, H, W, C_, hp, wp, _ptr(tokens), _stream())
    return tokens


def fusion_core(wts, B, pvec_dwi_sum, pvec_dce_sum, npix, mask_dwi, mask_dce, npix_mask, tok_dwi, tok_dce,
                gating, attn, lowres, gate, logits):
    _call("b200_fusion_core", None, C.byref(wts), B, _ptr(pvec_dwi_sum), _ptr(pvec_dce_sum), npix, _ptr(mask_dwi),
                                  _ptr(mask_dce), npix_mask, _ptr(tok_dwi), _ptr(tok_dce), _ptr(gating), _ptr(attn),
                                  _ptr(lowres), _ptr(gate), _ptr(logits), _stream())


def fusion_mix(p_dwi, p_dce, gating, lowres, gate, hp, wp, out):
    B, H, W, C_ = p_dwi.shape
    _call("b200_fusion_mix", None, _ptr(p_dwi), _ptr(p_dce), _ptr(gating), _ptr(lowres), _ptr(gate), B, H, W, C_, hp,
                                 wp, _ptr(out), _stream())
    return out


# ---------------------------------------------------------------------------------------------------------------
# fusion-head fine-tuning step (csrc/train_ops.cu); every tensor is fp32 and row-major
# ---------------------------------------------------------------------------------------------------------------
def _f32_rows(t, name):
    if t.dtype != torch.float32 or t.dim() != 2 or t.stride(1) != 1:
        raise B200NativeError(f"{name} must be a 2-D float32 tensor with unit column stride")
    return t


def sgemm(a, b, out, *, trans_a=False, trans_b=False, bias=None, res=None, res_div=1, pre=None, act=0, beta=0,
          split_k=1):
    """out = op(a) @ op(b) (+ bias, + res broadcast over res_div rows; pre <- value before GELU; beta=1 accumulates).
    a, b, out (and res) are 2-D fp32 tensors or row-strided views of them."""
    _f32_rows(a, "a"), _f32_rows(b, "b"), _f32_rows(out, "out")
    M, K = (a.shape[1], a.shape[0]) if trans_a else a.shape
    Kb, N = (b.shape[1], b.shape[0]) if trans_b else b.shape
    if K != Kb or tuple(out.shape) != (M, N):
        raise B200NativeError(f"sgemm shape mismatch: op(a) {M}x{K}, op(b) {Kb}x{N}, out {tuple(out.shape)}")
    if res is not None:
        _f32_rows(res, "res")
        if res.shape[1] != N or res.shape[0] * res_div != M:
            raise B200NativeError("sgemm residual shape mismatch")
    if pre is not None and (pre.shape != out.shape or pre.stride(0) != out.stride(0)):
        raise B200NativeError("sgemm pre-activation output must have the layout of out")
    if bias is not None and bias.numel() != N:
        raise B200NativeError("sgemm bias length mismatch")
    _call("b200_sgemm", (M, N, K, int(trans_a), int(trans_b)), _ptr(a), a.stride(0), int(trans_a), _ptr(b), b.stride(0), int(trans_b), _ptr(out),
          out.stride(0), M, N, K, _ptr(bias), _ptr(res), res.stride(0) if res is not None else 0, res_div, _ptr(pre),
          act, beta, split_k, _stream())
    return out


def colsum(x, out):
    """out[n] += sum_r x[r, n]."""
    _f32_rows(x, "x")
    if out.numel() != x.shape[1] or out.dtype != torch.float32:
        raise B200NativeError("colsum output mismatch")
    _call("b200_colsum", None, _ptr(x), x.stride(0), x.shape[0], x.shape[1], _ptr(out), _stream())
    return out


def mha_fwd(q, k, v, B, heads, probs, ctx):
    """q [B*Tq, C] and k / v [B*Tk, C] (row-strided views allowed, k and v with the same row stride)."""
    Tq, Tk, DH = q.shape[0] // B, k.shape[0] // B, q.shape[1] // heads
    if k.stride(0) != v.stride(0):
        raise B200NativeError("k and v must share a row stride")
    _call("b200_mha_fwd", None, _ptr(q), q.stride(0), _ptr(k), _ptr(v), k.stride(0), B, heads, Tq, Tk, DH,
          _ptr(probs), _ptr(ctx), ctx.stride(0), _stream())
    return probs, ctx


def mha_bwd(q, k, v, probs, dctx, B, heads, dq, dk, dv):
    Tq, Tk, DH = q.shape[0] // B, k.shape[0] // B, q.shape[1] // heads
    if k.stride(0) != v.stride(0) or dk.stride(0) != k.stride(0) or dv.stride(0) != k.stride(0) or \
            dq.stride(0) != q.stride(0):
        raise B200NativeError("mha_bwd gradients must have the layouts of q / k / v")
    _call("b200_mha_bwd", None, _ptr(q), q.stride(0), _ptr(k), _ptr(v), k.stride(0), _ptr(probs), _ptr(dctx),
          dctx.stride(0), B, heads, Tq, Tk, DH, _ptr(dq), _ptr(dk), _ptr(dv), _stream())
    return dq, dk, dv


def ln_fwd(x, w, b, eps, y, mean, rstd):
    R, C_ = x.shape
    _call("b200_ln_fwd", None, _ptr(x), R, C_, _ptr(w), _ptr(b), float(eps), _ptr(y), _ptr(mean), _ptr(rstd),
          _stream())
    return y


def ln_bwd(x, dy, dres, w, mean, rstd, dx, dyxhat):
    R, C_ = x.shape
    _call("b200_ln_bwd", None, _ptr(x), _ptr(dy), _ptr(dres), R, C_, _ptr(w), _ptr(mean), _ptr(rstd), _ptr(dx),
          _ptr(dyxhat), _stream())
    return dx


def gelu_bwd(pre, dg, out):
    _call("b200_gelu_bwd", None, _ptr(pre), _ptr(dg), pre.numel(), _ptr(out), _stream())
    return out


def head_loss(args, B):
    _call("b200_head_loss", None, C.byref(args), B, _stream())


def adamw(p, g, m, v, *, lr, betas, eps, weight_decay, step, grad_scale=1.0):
    for t in (p, g, m, v):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != p.numel():
            raise B200NativeError("adamw needs equally sized contiguous float32 buffers")
    _call("b200_adamw", None, _ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), float(lr), float(betas[0]),
          float(betas[1]), float(eps), float(weight_decay), int(step), float(grad_scale), _stream())


def mask_dot(f3, omega, out):
    """f3 NHWC bf16 [B,H,W,Cin] (contiguous), omega [B,Cin] fp32 -> out [B,H*W] fp32."""
    _bf16_map(f3, "f3")
    if not f3.is_contiguous():
        raise B200NativeError("mask_dot needs a contiguous NHWC map")
    B, H, W, Cin = f3.shape
    _call("b200_mask_dot", None, _ptr(f3), _ptr(omega), B, H * W, Cin, _ptr(out), _stream())
    return out


def mask_wsum(f3, dm, out):
    """out[b,:] = sum_p dm[b,p] * f3[b,p,:]."""
    if f3.dtype != torch.bfloat16 or not f3.is_contiguous():
        raise B200NativeError("mask_wsum needs a contiguous bfloat16 NHWC map")
    B, H, W, Cin = f3.shape
    _call("b200_mask_wsum", None, _ptr(f3), _ptr(dm), B, H * W, Cin, _ptr(out), _stream())
    return out


def mask_dice(D_dwi, D_dce, gating, u, lowres, pre_b, out_w, out_b, target, enc_dwi, enc_dce, H, W, Ho, Wo, hp, wp,
              scale, eps, loss_type, m_out, dm_out, q_out, dc0_out, loss_out):
    B, C_ = u.shape
    _call("b200_mask_dice", None, _ptr(D_dwi), _ptr(D_dce), _ptr(gating), _ptr(u), _ptr(lowres), _ptr(pre_b),
          _ptr(out_w), _ptr(out_b), pre_b.numel(), _ptr(target), _ptr(enc_dwi), _ptr(enc_dce), B, H, W, Ho, Wo, hp, wp, C_,
          float(scale), float(eps), int(loss_type), _ptr(m_out), _ptr(dm_out), _ptr(q_out), _ptr(dc0_out), _ptr(loss_out), _stream())


def mask_head_grads(dv, dc0, pre_w, pre_b, out_w, g_pre_w, g_pre_b, g_out_w, g_out_b):
    mid, C_ = pre_b.numel(), dv.numel()
    _call("b200_mask_head_grads", None, _ptr(dv), _ptr(dc0), _ptr(pre_w), _ptr(pre_b), _ptr(out_w), mid, C_,
          _ptr(g_pre_w), _ptr(g_pre_b), _ptr(g_out_w), _ptr(g_out_b), _stream())


def augment(x, theta, flips, out, fill=0.0):
    """x, out [B,C,H,W] fp32; theta [B,6] fp32 inverse affine matrices; flips [B] int32 (bit 0 horizontal, bit 1
    vertical) or None."""
    if x.dtype != torch.float32 or not x.is_contiguous() or out.shape != x.shape or not out.is_contiguous():
        raise B200NativeError("augment needs contiguous float32 [B,C,H,W] tensors of equal shape")
    B, C_, H, W = x.shape
    if theta.shape != (B, 6) or theta.dtype != torch.float32 or not theta.is_contiguous():
        raise B200NativeError("theta must be a contiguous float32 [B,6] tensor")
    if flips is not None and (flips.dtype != torch.int32 or flips.numel() != B):
        raise B200NativeError("flips must be an int32 [B] tensor")
    _call("b200_augment", None, _ptr(x), _ptr(out), B, C_, H, W, _ptr(theta), _ptr(flips), float(fill), _stream())
    return out
