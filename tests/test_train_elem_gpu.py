"""GPU: every C entry point of csrc/train_elem.cu, one launch at a time through the C ABI, against a plain fp64 restatement
of the same operation on the CPU (fp64 autograd for the backward passes), at the shapes where the kernels branch: ragged
row tails, strided views (ld > C), channel counts whose 8-channel groups do not divide the 256-thread CTA, every template
instantiation a dispatcher can pick.

Every reference is fed exactly what the kernel reads (bf16 maps rounded first, fp32 parameters as fp32).  Outputs are
compared element-wise with  |got - ref| <= rtol |ref| + atol S  where S is the sum of the absolute values of the terms
that make up the element (computed alongside the reference), rtol comes from the output's storage type and atol from the
longest fp32 accumulation chain the kernel runs for that element.  Outputs the kernel overwrites are pre-filled with NaN
(every element must be written), accumulated outputs with known values, and the padding columns of strided outputs with
a sentinel that must survive.

Not covered: the 64-bit index paths of map_scale_add / map_axpby (they need more than 2^30 16-byte vectors)."""
import math

import pytest
import torch
import torch.nn.functional as F

import b200path  # noqa: F401
import b200_native as nat

pytestmark = pytest.mark.gpu
DEV = "cuda"
D64 = torch.float64
U = 2.0 ** -24        # fp32 unit roundoff
BF = 2.0 ** -8        # rtol of a bf16-stored output (its unit roundoff: 8 significant bits)
F32 = 4 * U           # rtol of an fp32-stored output
E_ERF = 9e-5          # |erf_poly(z) - erf(z)| of the BatchNorm kernels' GELU (8.9e-5 on [0, 6], clamp included)
PAD = 776.0           # sentinel of the padding columns (exact in bf16)


# ------------------------------------------------------------------------------------------------------- helpers ----
def _g(seed):
    return torch.Generator().manual_seed(seed)


def _bf(t):
    """the bf16 value the kernel reads, as fp64"""
    return t.bfloat16().double()


def _f(t):
    """the fp32 value the kernel reads, as fp64"""
    return t.float().double()


_LIVE = []  # device tensors whose addresses were handed out: kept alive until the launch that reads them has run


def _p(t):
    if t is None:
        return None
    _LIVE.append(t)
    return t.data_ptr()


def _call(name, *args):
    nat._call(name, None, *args, nat._stream())
    torch.cuda.synchronize()
    _LIVE.clear()


def _map(vals, ld, fill=float("nan")):
    """[R, C] (bf16-exact) -> bf16 device buffer [R, ld] holding vals in its first C columns; the padding holds `fill`
    (NaN for inputs: a kernel that reads it produces non-finite output)."""
    R, C = vals.shape
    buf = torch.full((R, ld), fill, dtype=torch.bfloat16)
    buf[:, :C] = vals.bfloat16()
    return buf.to(DEV)


def _out_map(R, C, ld):
    """bf16 output buffer [R, ld]: NaN where the kernel must write, PAD in the padding it must leave alone"""
    buf = torch.full((R, ld), PAD, dtype=torch.bfloat16)
    buf[:, :C] = float("nan")
    return buf.to(DEV)


def _cols(buf, C):
    """the C used columns of a strided map, fp64 on the CPU; asserts the padding columns still hold the sentinel"""
    b = buf.cpu()
    if b.shape[1] > C and not (b[:, C:].float() == PAD).all():
        print("padding columns of a strided output were written")
        raise AssertionError("padding columns of a strided output were written")
    return b[:, :C].double()


def _dev(t, dtype=torch.float32):
    return t.to(dtype).to(DEV)


def _check(name, got, ref, bound):
    got = got.detach().double().cpu().reshape(ref.shape)
    ref = ref.detach().double()
    bound = torch.as_tensor(bound, dtype=D64).expand_as(ref)
    bad = ~torch.isfinite(got)
    if bad.any():
        print(f"{name}: {int(bad.sum())} elements not written or not finite")
        raise AssertionError(f"{name}: {int(bad.sum())} elements not written or not finite")
    err = (got - ref).abs()
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    worst = ratio.max().item()
    print(f"{name}: worst |got - ref| / bound = {worst:.3g}")
    if worst > 1:
        i = int(ratio.flatten().argmax())
        msg = (f"{name}: |got - ref| / bound = {worst:.3g} at flat index {i} of {tuple(ref.shape)}: got "
               f"{got.flatten()[i].item()!r} ref {ref.flatten()[i].item()!r} bound {bound.flatten()[i].item():.3g}")
        print(msg)
        raise AssertionError(msg)


def _ceil(a, b):
    return -(-a // b)


# --------------------------------------------------------------------------------------------- BatchNorm stats ------
@pytest.mark.parametrize("C,R,pad", [(8, 5003, 0), (24, 4099, 8), (40, 1237, 0), (96, 2051, 16), (512, 1000, 8),
                                     (2048, 37, 0)])
def test_bn_stats_vs_fp64(C, R, pad):
    """nn.BatchNorm2d batch sums: fp64 sum / sum of squares per channel, ACCUMULATED into the caller's buffers."""
    g = _g(C * 31 + R)
    z = _bf(torch.randn(R, C, generator=g) * 1.5 + 0.3)
    s0, q0 = torch.randn(C, generator=g, dtype=D64), torch.rand(C, generator=g, dtype=D64)
    sd, qd = s0.to(DEV), q0.to(DEV)
    _call("b200_bn_stats", _p(_map(z, C + pad)), R, C, C + pad, _p(sd), _p(qd))
    rows_par = 256 // (C // 8)
    grid = min(max(_ceil(R, rows_par * 16), 1), 148 * 4)
    L = _ceil(R, grid * rows_par)  # rows one thread sums in fp32 before the fp64 reduction
    _check("bn_stats sum", sd, s0 + z.sum(0), L * U * z.abs().sum(0))           # atol: fp32 chain of L terms
    _check("bn_stats sumsq", qd, q0 + (z * z).sum(0), L * U * (z * z).sum(0))


@pytest.mark.parametrize("count", [1, 7, 1000])
def test_bn_finalize_vs_fp64(count):
    """mean, 1/sqrt(biased var + eps) and the running-statistics update (unbiased variance, momentum) of
    nn.BatchNorm2d in training mode; count = 1 takes the unbiased-variance guard."""
    C, eps, mom = 37, 1e-5, 0.1
    g = _g(count)
    x = torch.randn(count, C, generator=g, dtype=D64) * 2 + 0.5
    x[:, 3] = 0.75                                   # a constant channel: var is exactly 0
    s, q = x.sum(0), (x * x).sum(0)
    q[5] = s[5] ** 2 / count * (1 - 1e-3)            # rounding made sumsq / n < mean^2: var clamps at 0
    rm0, rv0 = torch.randn(C, generator=g).float(), (torch.rand(C, generator=g) + 0.5).float()
    epsf, momf = _f(torch.tensor(eps)).item(), _f(torch.tensor(mom)).item()
    m = s / count
    v = (q / count - m * m).clamp_min(0)
    unb = v * count / (count - 1) if count > 1 else v
    refs = {"mean": m, "invstd": 1 / torch.sqrt(v + epsf),
            "running_mean": (1 - momf) * rm0.double() + momf * m, "running_var": (1 - momf) * rv0.double() + momf * unb}
    for with_running in (True, False):
        out = {k: torch.full((C,), math.nan, device=DEV) for k in ("mean", "invstd")}
        rm, rv = rm0.to(DEV), rv0.to(DEV)
        _call("b200_bn_finalize", _p(s.to(DEV)), _p(q.to(DEV)), C, float(count), eps, mom, _p(rm) if with_running else None,
              _p(rv) if with_running else None, _p(out["mean"]), _p(out["invstd"]))
        out.update(running_mean=rm, running_var=rv)
        for k, ref in refs.items():
            if with_running or not k.startswith("running"):
                _check(f"bn_finalize {k}", out[k], ref, F32 * ref.abs())     # fp64 arithmetic, one fp32 rounding
        if not with_running:
            assert torch.equal(rm.cpu(), rm0) and torch.equal(rv.cpu(), rv0)
    assert refs["invstd"][3].item() == 1 / math.sqrt(epsf) and refs["invstd"][5].item() == 1 / math.sqrt(epsf)


# ------------------------------------------------------------------------------------------ BatchNorm + activation --
def _act(y, act):
    return F.gelu(y) if act == 1 else (torch.relu(y) if act == 2 else y)


def _bn_launch_rows(R, C):
    """rows one thread walks in the BN kernels (bn_grid in train_elem.cu)"""
    rows_par = 256 // (C // 4)
    grid = min(max(_ceil(R, rows_par * 4), 1), 148 * 8)
    return _ceil(R, grid * rows_par)


def _bn_inputs(g, R, C, batch_stats, null, eps=1e-5):
    z = _bf(torch.randn(R, C, generator=g) * 1.5 + 0.3)
    gamma = (1 + 0.3 * torch.randn(C, generator=g)).float()
    beta = (0.2 * torch.randn(C, generator=g)).float()
    if batch_stats:
        mean = z.mean(0).float()
        invstd = (z.var(0, unbiased=False) + eps).rsqrt().float()
    else:
        mean, invstd = (0.3 + 0.2 * torch.randn(C, generator=g)).float(), (0.5 + torch.rand(C, generator=g)).float()
    par = {"mean": mean, "invstd": invstd, "gamma": gamma, "beta": beta}
    for k in null.split(","):
        if k:
            par[k] = None
    eff = {k: (_f(v) if v is not None else torch.full((C,), 1.0 if k in ("invstd", "gamma") else 0.0, dtype=D64))
           for k, v in par.items()}
    return z, par, eff


def _bn_ref_y(z, rs, eff, batch_stats, eps=1e-5):
    """y = bn(z) + res, fp64 (code/model_module.py:220-316 with nn.BatchNorm2d in training mode); with batch statistics
    the normalisation is differentiated through the batch mean / variance"""
    if batch_stats:
        mu = z.mean(0)
        xh = (z - mu) * (((z - mu) ** 2).mean(0) + eps).rsqrt()
    else:
        xh = (z - eff["mean"]) * eff["invstd"]
    return xh * eff["gamma"] + eff["beta"] + (rs if rs is not None else 0), xh


BN_CASES = [  # C, act, residual, pad, batch_stats, null parameters
    (24, 2, True, 8, 1, ""),
    (40, 1, False, 0, 1, ""),
    (64, 0, True, 16, 0, ""),
    (96, 1, True, 8, 0, "gamma,beta"),
    (16, 1, False, 0, 0, "mean,invstd"),
    (1024, 1, True, 8, 1, ""),
    (8, 2, False, 0, 1, "beta"),
]


@pytest.mark.parametrize("C,act,res,pad,batch_stats,null", BN_CASES)
def test_bn_act_fwd_bwd_vs_fp64(C, act, res, pad, batch_stats, null):
    """b200_bn_act_fwd: out = act(gamma (z - mean) invstd + beta + res);  b200_bn_act_bwd: dz, dres, dgamma += , dbeta +=
    (batch_stats = 1: through the batch statistics, pass 2 in place on dz; 0: fixed statistics, pass 2 only for
    dgamma / dbeta)."""
    R, ld = 611, C + pad
    g = _g(C * 10 + act)
    z, par, eff = _bn_inputs(g, R, C, batch_stats, null)
    rs = _bf(torch.randn(R, C, generator=g)) if res else None
    dA = _bf(torch.randn(R, C, generator=g))
    a = _f(eff["invstd"].float() * eff["gamma"].float())  # the kernel's folded per-channel scale (fp32)
    # |terms| of y = z a + (beta - mean a) + res
    S_y = (z * a).abs() + (eff["mean"] * a).abs() + eff["beta"].abs() + (rs.abs() if res else 0)
    y_fix, _ = _bn_ref_y(z, rs, eff, False)
    if act == 2:  # the ReLU kink: no gradient through elements whose sign the fp32 y cannot decide
        dA = torch.where(y_fix.abs() <= 1e-4 * S_y, torch.zeros_like(dA), dA)
    zd, rd, dAd = _map(z, ld), (_map(rs, ld) if res else None), _map(dA, ld)
    P = {k: (_dev(v) if v is not None else None) for k, v in par.items()}
    pargs = (_p(P["mean"]), _p(P["invstd"]), _p(P["gamma"]), _p(P["beta"]))
    out = _out_map(R, C, ld)
    _call("b200_bn_act_fwd", _p(zd), ld, _p(rd), ld, *pargs, act, 0.0, 0, R, C, _p(out), ld)
    out_ref = _act(y_fix, act)
    # atol: fp32 fold / fma / residual add (4 U on S_y), and the GELU's polynomial erf (0.5 |y| E_ERF)
    _check("bn_act_fwd out", _cols(out, C), out_ref, BF * out_ref.abs() + (4 * U + (E_ERF / 2 if act == 1 else 0)) * S_y)

    zr = z.clone().requires_grad_(True)
    rr = rs.clone().requires_grad_(True) if res else None
    y, xh = _bn_ref_y(zr, rr, eff, batch_stats)
    yy = y.detach().clone().requires_grad_(True)
    _act(yy, act).backward(dA)
    dY = yy.grad                                                   # gradient at y (= dres)
    y.backward(dY)
    xh = xh.detach()
    dz = _out_map(R, C, ld)
    dres = _out_map(R, C, ld) if res else None
    dg0, db0 = torch.randn(C, generator=g).float(), torch.randn(C, generator=g).float()
    dgd, dbd = dg0.to(DEV), db0.to(DEV)
    scratch = torch.empty(2 * C, dtype=D64, device=DEV)
    _call("b200_bn_act_bwd", _p(zd), ld, _p(rd), ld, *pargs, act, 0.0, 0, R, C, _p(dAd), ld, batch_stats, _p(scratch),
          _p(dz), ld, _p(dres), ld, _p(dgd), _p(dbd))
    L = _bn_launch_rows(R, C)
    # error of the kernel's dY = dA act'(y): polynomial erf and fp32 y (GELU'' <= 0.8); exact for identity / ReLU
    e_dY = dA.abs() * (E_ERF / 2 + 0.8 * 4 * U * S_y + 4 * U) if act == 1 else 2 * U * dY.abs()
    if res:
        _check("bn_act_bwd dres", _cols(dres, C), rr.grad, BF * rr.grad.abs() + e_dY)
    mu, inv = eff["mean"], eff["invstd"]
    # s1 = sum dY, s2 = (sum dY z - mu sum dY) invstd: fp32 chains of L rows, then fp64
    e_s1 = L * U * dY.abs().sum(0) + e_dY.sum(0)
    e_s2 = inv * (L * U * (dY * z).abs().sum(0) + mu.abs() * L * U * dY.abs().sum(0) + ((z.abs() + mu.abs()) * e_dY).sum(0))
    dgamma_ref, dbeta_ref = (dY * xh).sum(0), dY.sum(0)
    _check("bn_act_bwd dgamma", dgd, dg0.double() + dgamma_ref, F32 * (dg0.double().abs() + dgamma_ref.abs()) + e_s2)
    _check("bn_act_bwd dbeta", dbd, db0.double() + dbeta_ref, F32 * (db0.double().abs() + dbeta_ref.abs()) + e_s1)
    if batch_stats:
        k1, k2 = dbeta_ref / R, dgamma_ref / R
        # dz = a (dY - k1 - xhat k2): dY went through the bf16 map between the passes (BF), k1 / k2 carry the sums'
        # errors, the folded fp32 coefficients 4 U on every term
        bound = BF * zr.grad.abs() + a.abs() * (BF * dY.abs() + e_dY + e_s1 / R + xh.abs() * e_s2 / R +
                                               4 * U * (dY.abs() + k1.abs() + ((z.abs() + mu.abs()) * inv * k2).abs()))
    else:
        bound = BF * zr.grad.abs() + a.abs() * (e_dY + 2 * U * dY.abs())
    _check("bn_act_bwd dz", _cols(dz, C), zr.grad, bound)


def test_bn_act_dropout_mask_matches_between_forward_and_backward():
    """Dropout after the activation: read the keep mask off a forward whose output cannot be 0, then the residual /
    GELU forward, the fixed-statistics backward (exactly 0 where dropped) and the batch-statistics backward must use
    the same mask for the same seed; another seed draws another mask."""
    C, R, p, eps = 24, 1000, 0.3, 1e-5
    g = _g(3)
    d = _bf(0.25 + 1.75 * torch.rand(R // 2, C, generator=g))
    sgn = torch.where(torch.rand(R // 2, C, generator=g) < 0.5, -1.0, 1.0).double()
    z = torch.cat([d * sgn, -d * sgn])[torch.randperm(R, generator=g)]    # batch mean exactly 0, |z - mean| >= 0.25
    invstd = (z.var(0, unbiased=False) + eps).rsqrt().float()
    gamma = (0.5 + torch.rand(C, generator=g)).float()
    rs, dA = _bf(torch.randn(R, C, generator=g)), _bf(torch.randn(R, C, generator=g))
    mean = torch.zeros(C)
    zd, rd, dAd = _map(z, C), _map(rs, C), _map(dA, C)
    md, isd, gd = _dev(mean), _dev(invstd), _dev(gamma)
    a = _f(invstd * gamma)
    y0 = z * a
    S_y = y0.abs()

    def fwd(seed, act=0, res=None):
        out = _out_map(R, C, C)
        _call("b200_bn_act_fwd", _p(zd), C, _p(res), C, _p(md), _p(isd), _p(gd), None, act, p, seed, R, C, _p(out), C)
        return out.cpu()

    s1, s2 = 0x1234_5678_9ABC, 0x0FED_CBA9_8765
    outA = fwd(s1)
    keep = outA != 0
    rate = 1 - keep.double().mean().item()
    assert abs(rate - p) < 5 * math.sqrt(p * (1 - p) / (R * C)), rate
    ref = y0 * keep / (1 - p)
    _check("dropout fwd (act 0)", outA, ref, BF * ref.abs() + 4 * U * S_y * keep / (1 - p))
    assert torch.equal(fwd(s1), outA), "same seed, different output"
    other = fwd(s2) != 0
    assert (other != keep).double().mean().item() > 0.3, "another seed drew the same mask"
    y1 = y0 + rs
    ref = F.gelu(y1) * keep / (1 - p)
    S1 = (S_y + rs.abs()) * keep / (1 - p)
    _check("dropout fwd (GELU + residual)", fwd(s1, 1, rd), ref, BF * ref.abs() + (4 * U + E_ERF / 2) * S1)

    # fixed statistics, GELU, residual: dz = a dY and dres = dY, exactly 0 on the dropped elements
    yr = y1.clone().requires_grad_(True)
    (F.gelu(yr) * keep / (1 - p)).backward(dA)
    dY = yr.grad
    dz, dres = _out_map(R, C, C), _out_map(R, C, C)
    scratch = torch.empty(2 * C, dtype=D64, device=DEV)
    _call("b200_bn_act_bwd", _p(zd), C, _p(rd), C, _p(md), _p(isd), _p(gd), None, 1, p, s1, R, C, _p(dAd), C, 0,
          _p(scratch), _p(dz), C, _p(dres), C, None, None)
    e_dY = dA.abs() * keep / (1 - p) * (E_ERF / 2 + 0.8 * 4 * U * S1 + 4 * U)
    _check("dropout bwd dres", _cols(dres, C), dY, BF * dY.abs() + e_dY)
    _check("dropout bwd dz (fixed statistics)", _cols(dz, C), a * dY, BF * (a * dY).abs() + a.abs() * (e_dY + 2 * U * dY.abs()))
    assert (dres.cpu()[~keep] == 0).all() and (dz.cpu()[~keep] == 0).all()

    # batch statistics, identity: the whole dz through the statistics with the same mask
    zr = z.clone().requires_grad_(True)
    mu = zr.mean(0)
    xh = (zr - mu) * (((zr - mu) ** 2).mean(0) + eps).rsqrt()
    (xh * _f(gamma) * keep / (1 - p)).backward(dA)
    dz = _out_map(R, C, C)
    _call("b200_bn_act_bwd", _p(zd), C, None, C, _p(md), _p(isd), _p(gd), None, 0, p, s1, R, C, _p(dAd), C, 1,
          _p(scratch), _p(dz), C, None, C, None, None)
    L = _bn_launch_rows(R, C)
    dY = dA * keep / (1 - p)
    inv, xh = _f(invstd), xh.detach()
    k1, k2 = dY.sum(0) / R, (dY * xh).sum(0) / R
    e1 = L * U * dY.abs().sum(0) / R
    e2 = inv * L * U * (dY * z).abs().sum(0) / R
    bound = BF * zr.grad.abs() + a.abs() * (BF * dY.abs() + 2 * U * dY.abs() + e1 + xh.abs() * e2 +
                                           4 * U * (dY.abs() + k1.abs() + (z * inv * k2).abs()))
    _check("dropout bwd dz (batch statistics)", _cols(dz, C), zr.grad, bound)


# ---------------------------------------------------------------------------------------------- map helpers --------
@pytest.mark.parametrize("C,npix,pad,two", [(8, 1001, 0, True), (24, 777, 8, True), (40, 300, 0, False),
                                            (96, 517, 16, True), (512, 1000, 8, False), (512, 999, 0, True)])
def test_map_dot_vs_fp64(C, npix, pad, two):
    """out[b, c] = sum_p a[b,p,c] b[b,p,c]  (b NULL: channel sums), OVERWRITTEN"""
    B, ld = 3, C + pad
    g = _g(C + npix)
    a = _bf(torch.randn(B * npix, C, generator=g))
    b = _bf(torch.randn(B * npix, C, generator=g)) if two else None
    out = torch.full((B, C), math.nan, device=DEV)
    _call("b200_map_dot", _p(_map(a, ld)), ld, _p(_map(b, ld + 8)) if two else None, ld + 8, B, npix, C, _p(out))
    t = (a * b if two else a).view(B, npix, C)
    rows_par = 256 // (C // 8)
    L = _ceil(npix, rows_par) + rows_par  # a thread's fp32 chain over its rows, then the fp32 sum of the row partials
    _check("map_dot", out, t.sum(1), L * U * t.abs().sum(1))


@pytest.mark.parametrize("C,npix,B,pad", [(64, 300, 3, 8), (24, 300, 2, 0), (40, 333, 3, 16), (40, 5000, 2, 0),
                                          (8, 1, 65536, 0)])
def test_map_scale_add_every_instantiation_vs_fp64(C, npix, B, pad):
    """out = x * gate[b] + add[b] (+ out if accumulate), every (x, gate, add, accumulate) instantiation of the per-case
    kernel plus the generic kernel (gate / add not 16-byte aligned, or B > 65535).  C = 24 / 40 take the division
    path and a stride that is not a multiple of C / 8; the broadcast forms (x NULL) are what the C5 backward runs."""
    g = _g(C * 7 + npix + B)
    R, ld = B * npix, C + pad
    x = _bf(torch.randn(R, C, generator=g))
    gate, add = torch.randn(B, C, generator=g).float(), torch.randn(B, C, generator=g).float()
    o0 = _bf(torch.randn(R, C, generator=g))
    xd = _map(x, ld)
    combos = [(hx, hg, ha, ac) for hx in (0, 1) for hg in (0, 1) for ha in (0, 1) for ac in (0, 1)]
    if B > 65535:
        combos = [(1, 1, 1, 1), (0, 0, 1, 0), (1, 1, 0, 0)]
    for misaligned in ((False, True) if B <= 65535 else (False,)):
        for hx, hg, ha, ac in combos:
            if misaligned and not (hg or ha):
                continue
            off = 1 if misaligned else 0
            gbuf = torch.empty(B * C + 1, device=DEV)
            abuf = torch.empty(B * C + 1, device=DEV)
            gbuf[off:off + B * C] = gate.flatten().to(DEV)
            abuf[off:off + B * C] = add.flatten().to(DEV)
            out = _map(o0, ld, PAD) if ac else _out_map(R, C, ld)
            _call("b200_map_scale_add", _p(xd) if hx else None, ld, gbuf[off:].data_ptr() if hg else None,
                  abuf[off:].data_ptr() if ha else None, B, npix, C, _p(out), ld, ac)
            gr = _f(gate).repeat_interleave(npix, 0)
            ar = _f(add).repeat_interleave(npix, 0)
            xv = x if hx else torch.full_like(x, 1.0 if hg else 0.0)
            v = xv * (gr if hg else 1) + (ar if ha else 0)
            ref = (o0 if ac else 0) + v
            S = (xv * (gr if hg else 1)).abs() + (ar.abs() if ha else 0) + (o0.abs() if ac else 0)
            _check(f"map_scale_add x{hx} gate{hg} add{ha} acc{ac}{' misaligned' if misaligned else ''}",
                   _cols(out, C), ref, BF * ref.abs() + 3 * U * S)


@pytest.mark.parametrize("C,R,pad,two", [(24, 1001, 8, True), (64, 517, 0, False), (40, 77, 16, True)])
def test_map_axpby_vs_fp64(C, R, pad, two):
    """y = alpha a + beta b (b NULL: alpha a), strided bf16 maps"""
    g = _g(C + R)
    a, b = _bf(torch.randn(R, C, generator=g)), _bf(torch.randn(R, C, generator=g))
    alpha, beta = 0.75, -1.5
    y = _out_map(R, C, C + pad)
    _call("b200_map_axpby", _p(_map(a, C + pad)), C + pad, alpha, _p(_map(b, C)) if two else None, C, beta, R, C, _p(y),
          C + pad)
    ref = alpha * a + (beta * b if two else 0)
    _check("map_axpby", _cols(y, C), ref, BF * ref.abs() + 2 * U * ((alpha * a).abs() + ((beta * b).abs() if two else 0)))


@pytest.mark.parametrize("C,R,pad", [(8, 3001, 0), (40, 777, 8)])
def test_map_sumsq_accumulates_vs_fp64(C, R, pad):
    """code/train.py:1021-1030: sum of squares of a bf16 map ACCUMULATED into an fp64 scalar"""
    a = _bf(torch.randn(R, C, generator=_g(R)))
    out = torch.tensor([3.5], dtype=D64, device=DEV)
    _call("b200_map_sumsq", _p(_map(a, C + pad)), C + pad, R, C, _p(out))
    total = R * (C // 8)
    grid = min(max(_ceil(total, 256), 1), 148 * 4)
    L = 8 * _ceil(total, grid * 256)  # one thread's fp32 chain
    ref = 3.5 + (a * a).sum()
    _check("map_sumsq", out, ref.view(1), L * U * (a * a).sum().view(1))


# ---------------------------------------------------------------------------------------------- squeeze-excite ------
@pytest.mark.parametrize("C,M", [(40, 10), (512, 32)])
def test_se_fwd_bwd_vs_fp64(C, M):
    """code/model_module.py:25-43: gate = sigmoid(W2 gelu(W1 (sums / npix) + b1) + b2); backward from dgate to dpooled
    (of the MEAN-pooled vector), da2, da1 and h"""
    B, npix = 3, 49
    g = _g(C + M)
    sums = (torch.randn(B, C, generator=g) * npix).float()
    w1, b1 = (torch.randn(M, C, generator=g) / C ** 0.5).float(), (0.1 * torch.randn(M, generator=g)).float()
    w2, b2 = (torch.randn(C, M, generator=g) / M ** 0.5).float(), (0.1 * torch.randn(C, generator=g)).float()
    dgate = torch.randn(B, C, generator=g).float()
    W = [_dev(t) for t in (w1, b1, w2, b2)]
    pooled, gate = torch.full((B, C), math.nan, device=DEV), torch.full((B, C), math.nan, device=DEV)
    _call("b200_se_fwd", _p(_dev(sums)), B, C, M, npix, *[_p(t) for t in W], _p(pooled), _p(gate))
    inv = _f(torch.tensor(1.0 / npix)).item()
    pr = _f(sums) * inv
    _check("se_fwd pooled", pooled, pr, F32 * pr.abs())
    pv = _f(pooled.cpu()).requires_grad_(True)
    W1, B1, W2, B2 = (_f(t) for t in (w1, b1, w2, b2))
    a1 = pv @ W1.T + B1
    h = F.gelu(a1)
    gr = torch.sigmoid(h @ W2.T + B2)
    # |terms|: a1 <- |W1||p| + |b1|; h <- 1.13 S_a1; a2 <- |W2| S_h + |b2|; gate <- 0.25 S_a2
    S_a1 = pv.detach().abs() @ W1.abs().T + B1.abs()
    S_a2 = (1.13 * S_a1) @ W2.abs().T + B2.abs()
    L = C // 32 + M // 32 + 16  # lane-strided fp32 chains + warp trees + gelu / sigmoid
    _check("se_fwd gate", gate, gr.detach(), F32 * gr.abs().detach() + L * U * 0.25 * S_a2)
    dp, da2, da1, hh = (torch.full(s, math.nan, device=DEV) for s in ((B, C), (B, C), (B, M), (B, M)))
    _call("b200_se_bwd", _p(pooled), *[_p(t) for t in W], _p(_dev(dgate)), B, C, M, _p(dp), _p(da2), _p(da1), _p(hh))
    a1r = a1.detach().requires_grad_(True)
    a2r = (F.gelu(a1r) @ W2.T + B2).detach().requires_grad_(True)
    torch.sigmoid(a2r).backward(_f(dgate))
    (F.gelu(a1r) @ W2.T).backward(a2r.grad)
    gr.backward(_f(dgate))
    L2 = L + C + M  # + the sequential fp32 loops over C (da1) and M (dpooled)
    S_da2 = _f(dgate).abs() * (0.25 + 0.1 * S_a2)
    S_da1 = (S_da2 @ W2.abs()) * (1.13 + 0.8 * S_a1)
    _check("se_bwd h", hh, h.detach(), F32 * h.detach().abs() + L * U * 1.13 * S_a1)
    _check("se_bwd da2", da2, a2r.grad, F32 * a2r.grad.abs() + L * U * S_da2)
    _check("se_bwd da1", da1, a1r.grad, F32 * a1r.grad.abs() + L2 * U * S_da1)
    _check("se_bwd dpooled", dp, pv.grad, F32 * pv.grad.abs() + L2 * U * (S_da1 @ W1.abs()))


# ----------------------------------------------------------------------------------------- C -> 1 convolutions -----
@pytest.mark.parametrize("C,taps,H,W,pad", [(8, 9, 7, 5, 8), (16, 1, 9, 11, 0), (64, 9, 13, 7, 0), (128, 1, 5, 3, 8),
                                            (256, 9, 5, 9, 16), (512, 9, 7, 9, 8), (512, 1, 6, 3, 0)])
def test_convc1_fwd_bwd_vs_fp64(C, taps, H, W, pad):
    """code/model_module.py:100-125 (1-channel convolutions): out = conv(x, w) + bias (1x1 or 3x3, padding 1);
    backward dx (overwritten, then accumulated), dw / dbias accumulated across launches"""
    B, ld, k = 2, C + pad, (3 if taps == 9 else 1)
    g = _g(C + taps + H)
    x = _bf(torch.randn(B, H, W, C, generator=g))
    w = (torch.randn(1, C, k, k, generator=g) / (C * taps) ** 0.5).float()
    bias = torch.tensor([0.3]).float()
    xd, wd, bd = _map(x.view(-1, C), ld), _dev(w), _dev(bias)
    out = torch.full((B, H, W), math.nan, device=DEV)
    _call("b200_convc1_fwd", _p(xd), ld, B, H, W, C, taps, _p(wd), _p(bd), _p(out))
    xn = x.permute(0, 3, 1, 2)
    ref = F.conv2d(xn, _f(w), _f(bias), padding=k // 2)[:, 0]
    S = F.conv2d(xn.abs(), _f(w).abs(), padding=k // 2)[:, 0] + 0.3
    L = 8 + 5 + C // 256 + taps + 1  # lane chain of 8, shuffle tree, > 256-channel chain, tap sum, bias
    _check("convc1_fwd", out, ref, F32 * ref.abs() + L * U * S)

    dout = torch.randn(B, H, W, generator=g).float()
    xr, wr, br = xn.clone().requires_grad_(True), _f(w).requires_grad_(True), _f(bias).requires_grad_(True)
    F.conv2d(xr, wr, br, padding=k // 2).backward(_f(dout)[:, None])
    dx_ref = xr.grad.permute(0, 2, 3, 1).reshape(-1, C)
    S_dx = F.conv_transpose2d(_f(dout).abs()[:, None], _f(w).abs(), padding=k // 2).permute(0, 2, 3, 1).reshape(-1, C)
    dw0, db0 = torch.randn(C * taps, generator=g).float(), torch.tensor([0.25])
    dwd, dbd = dw0.to(DEV), db0.to(DEV)
    dx = _out_map(B * H * W, C, ld)
    for rep in range(2):
        prev = _cols(dx, C) if rep else 0
        _call("b200_convc1_bwd", _p(xd), ld, _p(_dev(dout)), B, H, W, C, taps, _p(wd), _p(dx), ld, rep, _p(dwd), _p(dbd))
        ref = prev + dx_ref
        _check(f"convc1_bwd dx (accumulate {rep})", _cols(dx, C), ref,
               BF * ref.abs() + (taps + 2) * U * (S_dx + (prev.abs() if rep else 0)))
    gl = min(C // 8, 32)
    nslots = 8 * (32 // gl)
    Ldw = _ceil(H * W, nslots) + nslots + 2 * B  # per-lane pixel chain, shared atomics of the slots, global atomics
    S_dw = F.conv2d(xn.abs().transpose(0, 1), _f(dout).abs()[None], padding=k // 2).transpose(0, 1).flatten() \
        if taps == 9 else (xn.abs() * _f(dout).abs()[:, None]).sum((0, 2, 3))
    ref_dw = dw0.double() + 2 * wr.grad.flatten()
    _check("convc1_bwd dw (2 launches)", dwd, ref_dw, F32 * ref_dw.abs() + 2 * Ldw * U * S_dw)
    ref_db = 0.25 + 2 * br.grad
    _check("convc1_bwd dbias (2 launches)", dbd, ref_db, F32 * ref_db.abs() + 2 * (2 * B + 4) * U * _f(dout).abs().sum())


# ------------------------------------------------------------------------------------------------ lift (1 -> N) ----
@pytest.mark.parametrize("N,P", [(8, 1001), (64, 4099), (128, 333)])
def test_lift_fwd_bwd_vs_fp64(N, P):
    """code/model_module.py:338 (Projector.proj[0] on r): z[p, n] = r[p] w[n]; dw[n] += sum_p dz r, dr[p] = sum_n dz w"""
    g = _g(N + P)
    r, w = torch.randn(P, generator=g).float(), torch.randn(N, generator=g).float()
    rd, wd = _dev(r), _dev(w)
    z = _out_map(P, N, N)
    _call("b200_lift_fwd", _p(rd), P, N, _p(wd), _p(z))
    ref = _f(r)[:, None] * _f(w)
    _check("lift_fwd", _cols(z, N), ref, BF * ref.abs())
    dz = _bf(torch.randn(P, N, generator=g))
    dw0 = torch.randn(N, generator=g).float()
    dw, dr = dw0.to(DEV), torch.full((P,), math.nan, device=DEV)
    _call("b200_lift_bwd", _p(_map(dz, N)), _p(rd), P, N, _p(wd), _p(dw), _p(dr))
    _check("lift_bwd dr", dr, dz @ _f(w), (N // 64 + 6) * U * (dz.abs() @ _f(w).abs()))
    grid = min(max(_ceil(P * 32, 256), 1), 148 * 4)
    L = _ceil(P, grid * 8) + 8 + grid  # a lane's pixel chain, shared atomics of 8 warps, global atomics
    ref = _f(dw0) + dz.T @ _f(r)
    _check("lift_bwd dw", dw, ref, F32 * ref.abs() + L * U * (dz.abs().T @ _f(r).abs()))


# ----------------------------------------------------------------------------------- mask-guided modulation --------
@pytest.mark.parametrize("C,P,pad", [(40, 333, 8), (512, 130, 0)])
def test_modulate_bwd_vs_fp64(C, P, pad):
    """code/model_module.py:97: y = f (1 + gamma A) -> df (overwritten), dA (overwritten), dgamma +="""
    g = _g(C + P)
    dy, f = _bf(torch.randn(P, C, generator=g)), _bf(torch.randn(P, C, generator=g))
    A, gamma = torch.rand(P, generator=g).float(), torch.tensor([0.7]).float()
    fr, Ar, gr = f.clone().requires_grad_(True), _f(A).requires_grad_(True), _f(gamma).requires_grad_(True)
    (fr * (1 + gr * Ar[:, None])).backward(dy)
    df, dA = _out_map(P, C, C + pad), torch.full((P,), math.nan, device=DEV)
    dgam = torch.tensor([0.5], device=DEV)
    _call("b200_modulate_bwd", _p(_map(dy, C + 8)), C + 8, _p(_map(f, C + pad)), C + pad, _p(_dev(A)), _p(_dev(gamma)), P, C,
          _p(df), C + pad, _p(dA), _p(dgam))
    _check("modulate_bwd df", _cols(df, C), fr.grad, BF * fr.grad.abs() + 3 * U * dy.abs() * (1 + 0.7 * _f(A)[:, None]))
    Lc = C // 32 + 6
    S_dot = (dy * f).abs().sum(1)
    _check("modulate_bwd dA", dA, Ar.grad, F32 * Ar.grad.abs() + Lc * U * 0.7 * S_dot)
    grid = min(max(_ceil(P * 32, 256), 1), 148 * 8)
    L = Lc + _ceil(P, grid * 8) + grid + 2
    ref = 0.5 + gr.grad
    _check("modulate_bwd dgamma", dgam, ref, F32 * ref.abs() + L * U * (S_dot * _f(A)).sum())


# ------------------------------------------------------------------------------------- mask attention backward -----
def _mask_attn_ref(m, wa, gnw, gnb, wb, bb, eps):
    """code/model_module.py:75-97 (oracle/model_oracle.py:103-112): A = clamp(sigmoid(conv1x1_K->1(gelu(
    GroupNorm(1, K)(conv1x1_1->K(mask))))), 1e-4, 1 - 1e-4)"""
    u = wa.view(1, -1, 1) * m[:, None, :]
    y = F.group_norm(u, 1, gnw, gnb, eps)
    s = (wb.view(1, -1, 1) * F.gelu(y)).sum(1) + bb
    return torch.clamp(torch.sigmoid(s), 1e-4, 1 - 1e-4), s


@pytest.mark.parametrize("K,npix,bb", [(16, 256, 0.2), (16, 300, 11.0), (5, 1000, -0.3), (32, 77, 0.1)])
def test_mask_attn_bwd_vs_fp64(K, npix, bb):
    """dm (OVERWRITTEN) and dwa, dgnw, dgnb, dwb, dbb (accumulated) of the mask attention; bb = 11 puts a share of the
    pixels in the clamped region, where their dA must not reach any gradient"""
    B, eps = 2, 1e-5
    g = _g(K + npix)
    m = torch.rand(B, npix, generator=g).float()
    wa, gnw, gnb = torch.randn(K, generator=g).float(), (1 + 0.3 * torch.randn(K, generator=g)).float(), \
        (0.2 * torch.randn(K, generator=g)).float()
    wb, bbt = (torch.randn(K, generator=g) * 2 / K ** 0.5).float(), torch.tensor([bb]).float()
    dA = torch.randn(B, npix, generator=g).float()
    P64 = [_f(t).requires_grad_(True) for t in (m, wa, gnw, gnb, wb, bbt)]
    A, s = _mask_attn_ref(*P64, eps)
    s = s.detach()
    edge = math.log((1 - 1e-4) / 1e-4)
    clamped = s.abs() > edge + 1e-3
    dA = torch.where((s.abs() - edge).abs() <= 1e-3, torch.zeros_like(dA), dA)  # undecidable at fp32: no gradient
    dA = torch.where(clamped, torch.full_like(dA, 1e6), dA)                    # must be stopped by the clamp
    if bb > 1:
        assert clamped.double().mean() > 0.05
    A.backward(_f(dA))
    grads0 = [torch.randn(K, generator=g).float() for _ in range(4)] + [torch.randn(1, generator=g).float()]
    gd = [t.to(DEV) for t in grads0]
    dm = torch.full((B, npix), math.nan, device=DEV)
    _call("b200_mask_attn_bwd", _p(_dev(m)), _p(_dev(dA)), B, npix, K, *[_p(_dev(t)) for t in (wa, gnw, gnb, wb, bbt)], eps,
          _p(dm), *[_p(t) for t in gd])
    # magnitudes: S_y of gn output, dxhat |terms|, GroupNorm backward rstd (|dxh| + mean|dxh| + |xh| mean|dxh xh|)
    mm, wa64, gw, gb, wb64 = (_f(t) for t in (m, wa, gnw, gnb, wb))
    u = wa64.view(1, -1, 1) * mm[:, None, :]
    mu = u.mean((1, 2), keepdim=True)
    rstd = (u.var((1, 2), unbiased=False, keepdim=True) + eps).rsqrt()
    xh = (u - mu) * rstd
    S_y = (u.abs() + mu.abs()) * rstd * gw.abs().view(1, -1, 1) + gb.abs().view(1, -1, 1)
    S_s = (wb64.abs().view(1, -1, 1) * 1.13 * S_y).sum(1) + abs(bb)
    a = torch.sigmoid(s)
    ds_mag = torch.where(clamped, torch.zeros_like(s), _f(dA).abs() * (a + a * a) * (1 + S_s))  # a (1 - a) = a - a^2
    dxh = ds_mag[:, None, :] * (wb64 * gw).abs().view(1, -1, 1) * (1.13 + 0.8 * S_y)
    n = K * npix
    T1, T2 = dxh.sum((1, 2), keepdim=True) / n, (dxh * xh.abs()).sum((1, 2), keepdim=True) / n
    S_du = rstd * (dxh + T1 + xh.abs() * T2)
    L = _ceil(npix, 256) * K + 4 * K + 64  # a thread's fp32 chain over its pixels and K, recompute of s, GN backward
    ref = P64[0].grad
    _check("mask_attn_bwd dm", dm, ref, F32 * ref.abs() + L * U * (S_du * wa64.abs().view(1, -1, 1)).sum(1))
    La = L + 256 + B  # + shared atomics of 256 threads and the global atomics of the B CTAs
    S_wa = (S_du * mm[:, None, :]).sum((0, 2))
    S_gw = (dxh / gw.abs().clamp_min(1e-30).view(1, -1, 1) * xh.abs()).sum((0, 2))
    S_gb = (dxh / gw.abs().clamp_min(1e-30).view(1, -1, 1)).sum((0, 2))
    S_wb = (ds_mag[:, None, :] * 1.13 * S_y).sum((0, 2))
    S_bb = ds_mag.sum().view(1)
    for name, t0, t, ref, S in zip(("dwa", "dgnw", "dgnb", "dwb", "dbb"), grads0, gd, [q.grad for q in P64[1:]],
                                   (S_wa, S_gw, S_gb, S_wb, S_bb)):
        ref = _f(t0) + ref
        _check(f"mask_attn_bwd {name}", t, ref, F32 * ref.abs() + La * U * S)


# ---------------------------------------------------------------------------------------------- stem backward -----
@pytest.mark.parametrize("C,N,stride,H,W,gate", [(1, 8, 1, 9, 7, True), (3, 64, 2, 34, 18, True), (8, 256, 2, 20, 36, False),
                                                 (9, 16, 1, 17, 16, True), (16, 128, 1, 12, 23, True),
                                                 (17, 32, 2, 22, 40, False), (32, 256, 1, 16, 17, True)])
def test_stem_bwd_vs_fp64(C, N, stride, H, W, gate):
    """first layer backward (b200_stem_ex, all outputs un-activated): z[b,p,n] = sum_c wcat[n,c] x[b,c,s p] gate[b,c];
    dwcat += (accumulated), dgate += ; CP = 8 / 16 / 32 instantiations, pixel counts that are not a multiple of 256"""
    B = 2
    g = _g(C * 100 + N + stride)
    x = torch.randn(B, C, H, W, generator=g).float()
    gt = (0.5 + torch.rand(B, C, generator=g)).float()
    w = (torch.randn(N, C, generator=g) / C ** 0.5).float()
    Ho, Wo = H // stride, W // stride
    dz = _bf(torch.randn(B, Ho * Wo, N, generator=g))
    xs = _f(x)[:, :, ::stride, ::stride].reshape(B, C, -1)           # [B, C, npix]
    gr, wr = _f(gt).requires_grad_(True), _f(w).requires_grad_(True)
    z = torch.einsum("nc,bcp->bpn", wr, xs * (gr[:, :, None] if gate else 1))
    z.backward(dz)
    dw0, dg0 = torch.randn(N, C, generator=g).float(), torch.randn(B, C, generator=g).float()
    dwd, dgd = dw0.to(DEV), dg0.to(DEV)
    _call("b200_stem_bwd", _p(_dev(x)), B, C, H, W, stride, _p(_dev(gt)) if gate else None, _p(dz.bfloat16().to(DEV)), N,
          _p(_dev(w)), _p(dwd), _p(dgd))
    npix = Ho * Wo
    S_dw = torch.einsum("bpn,bcp->nc", dz.abs(), xs.abs() * (_f(gt).abs()[:, :, None] if gate else 1))
    L = npix + B + 2  # a thread's chain over the pixels of its case, the gate product, the atomics of the B CTAs
    ref = _f(dw0) + wr.grad
    _check("stem_bwd dwcat", dwd, ref, F32 * ref.abs() + L * U * S_dw)
    S_dg = torch.einsum("bpn,nc,bcp->bc", dz.abs(), _f(w).abs(), xs.abs())
    Lg = N + _ceil(npix, 256) + 5 + 8 + 1  # t = sum_n (chain N), a thread's tiles, warp tree, 8 warps' atomics, global
    ref = _f(dg0) + (gr.grad if gate else torch.einsum("bpn,nc,bcp->bc", dz, _f(w), xs))
    _check("stem_bwd dgate", dgd, ref, F32 * ref.abs() + Lg * U * S_dg)


# --------------------------------------------------------------------------------------------- classifier head ----
@pytest.mark.parametrize("C,K,normalize", [(200, 1, 1), (200, 2, 0), (300, 16, 1), (64, 7, 1), (520, 16, 0)])
def test_cls_head_bwd_vs_fp64(C, K, normalize):
    """code/model_module.py:355-369: logits = W (v / max(|v|, 1e-12)) + b (normalize) or W v + b; dfcw, dfcb accumulated,
    dpooled overwritten; case 0 has a zero pooled vector (the 1e-12 clamp of the norm)"""
    B = 3
    g = _g(C + K + normalize)
    v = torch.randn(B, C, generator=g).float()
    v[0] = 0
    w, dl = (torch.randn(K, C, generator=g) / C ** 0.5).float(), torch.randn(B, K, generator=g).float()
    V, Wm, DL = _f(v), _f(w), _f(dl)
    nrm = V.norm(dim=1, keepdim=True)
    epsf = _f(torch.tensor(1e-12)).item()
    nrm_c = nrm.clamp_min(epsf) if normalize else torch.ones_like(nrm)
    u = V / nrm_c
    gg = DL @ Wm
    if normalize:  # d(v / max(|v|, eps)): (g - u <g, u>) / |v| above the clamp, g / eps below it
        dp_ref = torch.where(nrm > epsf, (gg - u * (gg * u).sum(1, keepdim=True)) / nrm_c, gg / epsf)
    else:
        dp_ref = gg
    dW0, db0 = torch.randn(K, C, generator=g).float(), torch.randn(K, generator=g).float()
    dWd, dbd, dpd = dW0.to(DEV), db0.to(DEV), torch.full((B, C), math.nan, device=DEV)
    _call("b200_cls_head_bwd", _p(_dev(v)), _p(_dev(dl)), _p(_dev(w)), B, C, K, normalize, _p(dWd), _p(dbd), _p(dpd))
    ref = _f(dW0) + DL.T @ u
    L = C // 256 + 8 + B  # norm: a thread's chain + fp64 tree; the atomics of B CTAs
    _check("cls_head_bwd dfcw", dWd, ref, F32 * ref.abs() + L * U * (DL.abs().T @ u.abs()))
    ref = _f(db0) + DL.sum(0)
    _check("cls_head_bwd dfcb", dbd, ref, F32 * ref.abs() + (B + 1) * U * DL.abs().sum(0))
    Sg = DL.abs() @ Wm.abs()
    S = (Sg + normalize * u.abs() * (Sg * u.abs()).sum(1, keepdim=True)) / nrm_c
    _check("cls_head_bwd dpooled", dpd, dp_ref, F32 * dp_ref.abs() + (K + L + C // 256 + 8) * U * S)


# ------------------------------------------------------------------------------------------------------ losses -----
@pytest.mark.parametrize("K,smoothing,gamma,weighted", [(2, 0.0, 0.0, False), (2, 0.1, 2.0, True), (5, 0.2, 1.0, True),
                                                        (16, 0.05, 2.0, False), (16, 0.1, 0.0, True)])
def test_focal_loss_vs_fp64(K, smoothing, gamma, weighted):
    """LabelSmoothing + Soft(Weighted)FocalLoss (code/loss.py:133-213): loss += scale sum_b l_b, dlogits = scale dl/dz;
    logits up to +-30"""
    B, scale = 70, 1.0 / 70
    g = _g(K * 10 + int(gamma * 4))
    z = (torch.randn(B, K, generator=g) * 3).float()
    z[0, 0], z[1, -1], z[2, :] = 30.0, -30.0, torch.linspace(-30, 30, K)
    lab = torch.randint(0, K, (B,), generator=g)
    cw = (0.5 + torch.rand(K, generator=g)).float() if weighted else None
    zr = _f(z).requires_grad_(True)
    lp = F.log_softmax(zr, 1)
    t = torch.full((B, K), smoothing / (K - 1), dtype=D64)
    t[torch.arange(B), lab] = 1 - smoothing
    t = _f(t)  # the kernel's fp32 targets
    wk = _f(cw) if weighted else torch.ones(K, dtype=D64)
    fw = (1 - lp.exp()).clamp_min(0) ** gamma
    lb = -(t * wk * fw * lp).sum(1)
    (scale * lb.sum()).backward()
    loss, dl = torch.tensor([0.5], device=DEV), torch.full((B, K), math.nan, device=DEV)
    _call("b200_focal_loss", _p(_dev(z)), _p(lab.to(DEV)), B, K, smoothing, gamma, _p(_dev(cw)) if weighted else None, scale,
          _p(loss), _p(dl))
    # fp32 log-softmax: |error of log p| <= 2 U (|z| + |lse|) + K U; everything else a few roundings of the terms
    lse = torch.logsumexp(_f(z), 1, keepdim=True)
    E = (4 * K + 8) * U + 2 * U * (_f(z).abs().max(1, keepdim=True)[0] + lse.abs())
    S = scale * (t * wk).abs().sum(1, keepdim=True) * (1 + lp.detach().abs()).max(1, keepdim=True)[0] * (1 + gamma) ** 2
    _check("focal_loss dlogits", dl, zr.grad, F32 * zr.grad.abs() + E * S)
    ref = 0.5 + scale * lb.detach().sum()
    _check("focal_loss loss", loss, ref.view(1), F32 * ref.abs() + (E * S).sum() + (B // 32 + 6) * U * scale * lb.abs().sum())


@pytest.mark.parametrize("n,empty", [(256, False), (1000, True), (4099, False)])
def test_dice_loss_vs_fp64(n, empty):
    """SoftDiceLoss (code/loss.py:45-62): loss += scale sum_b (1 - (2 I + eps) / (U + eps)), dlogits overwritten; case 0
    has an all-zero target when `empty`"""
    B, eps, scale = 3, 1.0, 0.5
    g = _g(n)
    z = (torch.randn(B, n, generator=g) * 2).float()
    tg = (torch.rand(B, n, generator=g) < 0.3).float()
    if empty:
        tg[0] = 0
    zr = _f(z).requires_grad_(True)
    p = torch.sigmoid(zr)
    T = _f(tg)
    dice = 1 - (2 * (p * T).sum(1) + eps) / (p.sum(1) + T.sum(1) + eps)
    (scale * dice.sum()).backward()
    loss, dl = torch.tensor([0.25], device=DEV), torch.full((B, n), math.nan, device=DEV)
    _call("b200_dice_loss", _p(_dev(z)), _p(_dev(tg)), B, n, eps, scale, _p(loss), _p(dl))
    L = _ceil(n, 256) + 16  # a thread's fp32 chain, then fp64 trees and the fp32 fraction
    den = (p.sum(1) + T.sum(1) + eps).detach()[:, None]
    # p (1 - p) = p - p^2 is formed from the fp32 sigmoid: near saturation its error is ~U p, not ~U p (1 - p)
    S = scale * (2 * T + 2 * (p * T).sum(1, keepdim=True).detach() / den + 1) / den * (p + p * p).detach()
    _check("dice_loss dlogits", dl, zr.grad, F32 * zr.grad.abs() + L * U * S)
    ref = 0.25 + scale * dice.detach().sum()
    _check("dice_loss loss", loss, ref.view(1), F32 * ref.abs() + L * U * scale * 2 * B)


@pytest.mark.parametrize("h,w,ratio,two", [(16, 12, 1, False), (16, 12, 2, True), (8, 6, 4, False), (10, 7, 4, True)])
def test_recon_loss_vs_fp64(h, w, ratio, two):
    """code/train.py:1041-1048, :446-454 (oracle/train_oracle.py:114-129): Charbonnier between sigmoid(bilinear-up r)
    and clamp(0,1) of the channel mean of x (and x2); loss +=, dr overwritten"""
    B, C, C2, eps = 2, 3, 2, 1e-3
    H, W = h * ratio, w * ratio
    scale = 1.0 / (B * H * W)
    g = _g(h * ratio + two)
    r = torch.randn(B, h, w, generator=g).float()
    x = (torch.rand(B, C, H, W, generator=g) * 1.4 - 0.2).float()
    x2 = (torch.rand(B, C2, H, W, generator=g) * 1.4 - 0.2).float() if two else None
    rr = _f(r).requires_grad_(True)
    up = F.interpolate(rr[:, None], size=(H, W), mode="bilinear", align_corners=False)[:, 0]
    tgt = (torch.cat([_f(x), _f(x2)], 1) if two else _f(x)).mean(1).clamp(0, 1)
    lossr = scale * torch.sqrt((torch.sigmoid(up).clamp(0, 1) - tgt) ** 2 + eps ** 2).sum()
    lossr.backward()
    loss, dr = torch.tensor([0.125], device=DEV), torch.full((B, h, w), math.nan, device=DEV)
    _call("b200_recon_loss", _p(_dev(r)), B, h, w, _p(_dev(x)), C, _p(_dev(x2)) if two else None, C2 if two else 0, H, W, eps,
          scale, _p(loss), _p(dr))
    # per output pixel: the fp32 bilinear value carries ~4 U (|v| + 1), d = s - t ~4 U (|s| + |t|), and the gradient
    # scale (d / e) s (1 - s) moves by up to eps^2 / e^3 per unit of d; dr gathers the output pixels through the
    # bilinear weights (fp32 shared atomics: up to 4 ratio^2 of them)
    v = up.detach()
    sg = torch.sigmoid(v)
    e = torch.sqrt((sg - tgt) ** 2 + eps ** 2)
    cond = scale * (sg + sg * sg) * (1 + (eps ** 2 / e ** 3) * (sg + tgt.abs() + v.abs() + 1))  # s (1 - s) = s - s^2
    r0 = torch.zeros(B, h, w, dtype=D64, requires_grad=True)
    F.interpolate(r0[:, None], size=(H, W), mode="bilinear", align_corners=False)[:, 0].backward(cond)
    L = 4 * ratio * ratio + 32
    _check("recon_loss dr", dr, rr.grad, F32 * rr.grad.abs() + L * U * r0.grad)
    ref = 0.125 + lossr.detach()
    Ll = _ceil(H * W, 256) + 32
    _check("recon_loss loss", loss, ref.view(1), F32 * ref.abs() + Ll * U * scale * (e + sg + tgt.abs() + v.abs() + 1).sum())


def test_mimic_loss_vs_fp64():
    """code/train.py:1033-1038 (oracle/train_oracle.py:132-136): loss += scale sum_b (1 - clamp(cos)), ds overwritten
    (teacher detached); case 2 is parallel to its teacher (outside the clamp: no gradient)"""
    B, n, scale = 3, 8 * 1001, 0.5
    g = _g(11)
    s = _bf(torch.randn(B, n, generator=g))
    t = _bf(torch.randn(B, n, generator=g) + 0.5 * s)
    s[2] = t[2] * 0.5                              # exactly parallel: cos = 1 > 1 - 1e-6
    sr = s.clone().requires_grad_(True)
    cos = (F.normalize(sr, dim=1) * F.normalize(t, dim=1)).sum(1)
    lossr = scale * (1 - cos.clamp(-1 + 1e-6, 1 - 1e-6)).sum()
    lossr.backward()
    loss, ds = torch.tensor([0.0], device=DEV), _out_map(B, n, n)
    _call("b200_mimic_loss", _p(_map(s, n)), _p(_map(t, n)), B, n, scale, _p(loss), _p(ds))
    L = _ceil(n, 256) + 16
    ns, nt = s.norm(dim=1, keepdim=True), t.norm(dim=1, keepdim=True)
    S = scale * (t.abs() / (ns * nt) + s.abs() / ns ** 2)
    _check("mimic_loss ds", _cols(ds, n), sr.grad, BF * sr.grad.abs() + L * U * S)
    assert (ds.cpu()[2] == 0).all()
    ref = lossr.detach()
    _check("mimic_loss loss", loss, ref.view(1), F32 * ref.abs() + L * U * scale * B)


@pytest.mark.parametrize("B,npix,C", [(4, 49, 64), (6, 300, 24)])
def test_mimic_pairs_vs_fp64(B, npix, C):
    """code/train_fusion.py:287-296: cases (0, 1) and (2, 3) as (student, teacher) pairs, cosine per CHANNEL over the
    pixels, averaged; dmap is zero everywhere except the student cases 0 and 2"""
    scale = 0.7
    g = _g(B + npix)
    m = _bf(torch.randn(B, npix, C, generator=g))
    mr = m.clone().requires_grad_(True)
    terms = []
    for i in (0, 2):
        s, t = mr[i], m[i + 1]
        cos = (F.normalize(s, dim=0) * F.normalize(t, dim=0)).sum(0)
        terms.append((1 - cos.clamp(-1 + 1e-6, 1 - 1e-6)).mean())
    lossr = scale * (terms[0] + terms[1]) / 2
    lossr.backward()
    loss, dmap = torch.tensor([0.0], device=DEV), torch.full((B, npix, C), math.nan, dtype=torch.bfloat16, device=DEV)
    _call("b200_mimic_pairs", _p(m.bfloat16().to(DEV)), B, npix, C, scale, _p(loss), _p(dmap))
    L = npix + 16  # a thread's fp32 chain over the pixels of its channel
    ns = m.norm(dim=1, keepdim=True)
    S = scale * 0.5 / C * (m.roll(-1, 0).abs() / (ns * ns.roll(-1, 0)) + m.abs() / ns ** 2)
    got = dmap.cpu().double()
    _check("mimic_pairs dmap", got, mr.grad, BF * mr.grad.abs() + L * U * S)
    assert (got[[1, 3]] == 0).all() and (got[4:] == 0).all()
    ref = lossr.detach()
    _check("mimic_pairs loss", loss, ref.view(1), F32 * ref.abs() + L * U * scale * 2)


# ------------------------------------------------------------------------------------------------- fusion head -----
@pytest.mark.parametrize("C,masks", [(64, True), (40, False)])
def test_gating_fwd_bwd_and_fused_pool_vs_fp64(C, masks):
    """GatingAttention (code/model_module.py:745-780): gx = [pvec_dwi, pvec_dce, mean(mask_dwi), mean(mask_dce)],
    alpha = softmax(W gx + b); backward to dgl, dgx, and the per-channel-SUM gradients; fused_pool:
    alpha0 pvec_d + alpha1 pvec_c + sum_t up[t] lowres[t]"""
    B, npix, npm, T = 3, 49, 300, 4
    g = _g(C + masks)
    sd, sc = (torch.randn(B, C, generator=g) * 7).float(), (torch.randn(B, C, generator=g) * 7).float()
    md, mc = torch.rand(B, npm, generator=g).float(), torch.rand(B, npm, generator=g).float()
    D = 2 * C + (2 if masks else 0)
    w, b = (torch.randn(2, D, generator=g) / D ** 0.5).float(), (0.1 * torch.randn(2, generator=g)).float()
    inv = _f(torch.tensor(1.0 / npix)).item()
    gxr = torch.cat([_f(sd) * inv, _f(sc) * inv] + ([_f(md).mean(1, keepdim=True), _f(mc).mean(1, keepdim=True)] if masks else []), 1)
    gxr.requires_grad_(True)
    alpha_r = torch.softmax(gxr @ _f(w).T + _f(b), 1)
    gx, alpha = torch.full((B, D), math.nan, device=DEV), torch.full((B, 2), math.nan, device=DEV)
    _call("b200_gating_fwd", _p(_dev(sd)), _p(_dev(sc)), B, C, npix, _p(_dev(md)) if masks else None,
          _p(_dev(mc)) if masks else None, npm, _p(_dev(w)), _p(_dev(b)), _p(gx), _p(alpha))
    _check("gating_fwd gx", gx, gxr.detach(), F32 * gxr.detach().abs() + (_ceil(npm, 256) + 12) * U * gxr.detach().abs())
    L = _ceil(D, 256) + 16
    S_l = (gxr.detach().abs() @ _f(w).abs().T + _f(b).abs()).sum(1, keepdim=True)
    _check("gating_fwd alpha", alpha, alpha_r.detach(), F32 * alpha_r.detach().abs() + L * U * S_l)
    dal = torch.randn(B, 2, generator=g).float()
    ar = _f(alpha.cpu())                          # the backward starts from the kernel's alpha (what it is handed)
    dgl_ref = ar * (_f(dal) - (ar * _f(dal)).sum(1, keepdim=True))
    dgx_ref = dgl_ref @ _f(w)
    dgl, dgx = torch.full((B, 2), math.nan, device=DEV), torch.full((B, D), math.nan, device=DEV)
    dpd, dpc = torch.full((B, C), math.nan, device=DEV), torch.full((B, C), math.nan, device=DEV)
    _call("b200_gating_bwd", _p(alpha), _p(_dev(dal)), _p(_dev(w)), B, C, D, npix, _p(dgl), _p(dgx), _p(dpd), _p(dpc))
    S_g = ar * (_f(dal).abs() + (ar * _f(dal)).abs().sum(1, keepdim=True))
    _check("gating_bwd dgl", dgl, dgl_ref, F32 * dgl_ref.abs() + 8 * U * S_g)
    S_x = S_g @ _f(w).abs()
    _check("gating_bwd dgx", dgx, dgx_ref, F32 * dgx_ref.abs() + 10 * U * S_x)
    _check("gating_bwd dpv_d", dpd, dgx_ref[:, :C] * inv, F32 * dgx_ref[:, :C].abs() * inv + 12 * U * S_x[:, :C] * inv)
    _check("gating_bwd dpv_c", dpc, dgx_ref[:, C:2 * C] * inv,
           F32 * dgx_ref[:, C:2 * C].abs() * inv + 12 * U * S_x[:, C:2 * C] * inv)

    lowres, up = torch.randn(B, T, C, generator=g).float(), torch.rand(T, generator=g).float()
    A = _f(alpha.cpu())
    for with_low in (True, False):
        out = torch.full((B, C), math.nan, device=DEV)
        _call("b200_fused_pool", _p(_dev(sd)), _p(_dev(sc)), B, C, npix, _p(alpha), _p(_dev(lowres)) if with_low else None,
              _p(_dev(up)), T, _p(out))
        ref = (A[:, :1] * _f(sd) + A[:, 1:] * _f(sc)) * inv
        S = (A[:, :1] * _f(sd).abs() + A[:, 1:] * _f(sc).abs()) * inv
        if with_low:
            ref = ref + torch.einsum("t,btc->bc", _f(up), _f(lowres))
            S = S + torch.einsum("t,btc->bc", _f(up).abs(), _f(lowres).abs())
        _check(f"fused_pool (lowres {with_low})", out, ref, F32 * ref.abs() + (T + 6) * U * S)


@pytest.mark.parametrize("H,W,C,Hp,Wp", [(14, 14, 64, 7, 7), (12, 10, 24, 3, 5), (10, 15, 40, 3, 5)])
def test_fusion_mix_bwd_both_phases_vs_fp64(H, W, C, Hp, Wp):
    """backward of fused = alpha0 p_dwi + alpha1 p_dce + bilinear_up(lowres): phase 0 dalpha +=, dlowres += ; phase 1
    dp_m = alpha_m dfused + dtok_m[bin] + dpvec_m (overwritten); dtok with H % Hp != 0 is rejected with -4"""
    B = 3
    g = _g(H * W + C)
    npix, T = H * W, Hp * Wp
    df, pd_, pc_ = (_bf(torch.randn(B, npix, C, generator=g)) for _ in range(3))
    alpha = torch.softmax(torch.randn(B, 2, generator=g), 1).float()
    low = torch.zeros(B, T, C, dtype=D64, requires_grad=True)
    al = _f(alpha).requires_grad_(True)
    upm = F.interpolate(low.view(B, Hp, Wp, C).permute(0, 3, 1, 2), size=(H, W), mode="bilinear", align_corners=False)
    fused = al[:, 0, None, None] * pd_ + al[:, 1, None, None] * pc_ + upm.permute(0, 2, 3, 1).reshape(B, npix, C)
    fused.backward(df)
    dal0, dlow0 = torch.randn(B, 2, generator=g).float(), torch.randn(B, T, C, generator=g).float()
    dald, dlowd = dal0.to(DEV), dlow0.to(DEV)
    dfd = df.bfloat16().to(DEV)
    _call("b200_fusion_mix_bwd", _p(dfd), _p(pd_.bfloat16().to(DEV)), _p(pc_.bfloat16().to(DEV)), None, B, H, W, C, Hp, Wp,
          _p(dald), _p(dlowd), None, None, None, None, None, None, 0)
    slabs = min(max(_ceil(148 * 2, B), 1), 16)
    L = _ceil(_ceil(npix, slabs) * (C // 8), 256) * 8 + 12 + slabs  # a thread's fp32 chain, fp64 tree, atomics
    S_a = torch.stack([(df * pd_).abs().sum((1, 2)), (df * pc_).abs().sum((1, 2))], 1)
    ref = _f(dal0) + al.grad
    _check("fusion_mix_bwd dalpha", dald, ref, F32 * ref.abs() + L * U * S_a)
    l0 = torch.zeros(B, T, C, dtype=D64, requires_grad=True)
    F.interpolate(l0.view(B, Hp, Wp, C).permute(0, 3, 1, 2), size=(H, W), mode="bilinear",
                  align_corners=False).permute(0, 2, 3, 1).reshape(B, npix, C).backward(df.abs())
    S_l = l0.grad                                   # sum_p |U[p, t] dfused[p, c]|
    ref = _f(dlow0) + low.grad
    Ll = 4 * _ceil(npix, T) + 8 + slabs  # the shared-memory atomics of one token's pixels, the global ones of the slabs
    _check("fusion_mix_bwd dlowres", dlowd, ref, F32 * ref.abs() + Ll * U * S_l)

    dtd, dtc = torch.randn(B, T, C, generator=g).float(), torch.randn(B, T, C, generator=g).float()
    dvd, dvc = torch.randn(B, C, generator=g).float(), torch.randn(B, C, generator=g).float()
    ok = H % Hp == 0 and W % Wp == 0
    dpd, dpc = torch.full((B, npix, C), math.nan, dtype=torch.bfloat16, device=DEV), \
        torch.full((B, npix, C), math.nan, dtype=torch.bfloat16, device=DEV)
    args = (_p(dfd), None, None, _p(_dev(alpha)), B, H, W, C, Hp, Wp, None, None, _p(_dev(dtd)), _p(_dev(dtc)),
            _p(_dev(dvd)), _p(_dev(dvc)), _p(dpd), _p(dpc), 1, nat._stream())
    rc = nat.lib().b200_fusion_mix_bwd(*args)
    if not ok:
        assert rc == -4
        args = args[:12] + (None, None) + args[14:]   # without dtok every shape is accepted
        assert nat.lib().b200_fusion_mix_bwd(*args) == 0
    else:
        assert rc == 0
    oy = torch.arange(H) * Hp // H
    ox = torch.arange(W) * Wp // W
    tok = (oy[:, None] * Wp + ox[None, :]).flatten()
    A = _f(alpha)
    for m, (got, dt, dv) in enumerate(((dpd, dtd, dvd), (dpc, dtc, dvc))):
        ref = A[:, m, None, None] * df + _f(dv)[:, None, :]
        S = (A[:, m, None, None] * df).abs() + _f(dv).abs()[:, None, :]
        if ok:
            ref = ref + _f(dt)[:, tok, :]
            S = S + _f(dt).abs()[:, tok, :]
        _check(f"fusion_mix_bwd dp{m}", got.cpu().double(), ref, BF * ref.abs() + 3 * U * S)


# ---------------------------------------------------------------------------------------------- small helpers ------
@pytest.mark.parametrize("H,W,C", [(7, 5, 24), (4, 4, 64)])
def test_up2_bwd_vs_fp64(H, W, C):
    """2x2 replication backward: din[b,h,w,c] = sum of the four replicas of dout (overwritten)"""
    B = 2
    dout = _bf(torch.randn(B, 2 * H, 2 * W, C, generator=_g(H * W + C)))
    din = torch.full((B, H, W, C), math.nan, dtype=torch.bfloat16, device=DEV)
    _call("b200_up2_bwd", _p(dout.bfloat16().to(DEV)), B, H, W, C, _p(din))
    ref = dout.view(B, H, 2, W, 2, C).sum((2, 4))
    _check("up2_bwd", din.cpu().double(), ref, BF * ref.abs() + 3 * U * dout.abs().view(B, H, 2, W, 2, C).sum((2, 4)))


def test_row_bcast_and_vec_axpby_vs_fp64():
    """row_bcast: out[b, i] = v[b * stride] * scale (overwritten); vec_axpby: y = alpha a + beta y, with beta = 0 the old
    y is not read (a NaN there does not leak)"""
    B, n, stride = 3, 1001, 5
    g = _g(1)
    v = torch.randn(B * stride, generator=g).float()
    out = torch.full((B, n), math.nan, device=DEV)
    _call("b200_row_bcast", _p(_dev(v)), stride, 0.3, B, n, _p(out))
    ref = (_f(v)[::stride] * _f(torch.tensor(0.3)).item())[:, None].expand(B, n)
    _check("row_bcast", out, ref, U * ref.abs())
    N = 300_001
    a, y0 = torch.randn(N, generator=g).float(), torch.randn(N, generator=g).float()
    y = y0.to(DEV)
    _call("b200_vec_axpby", _p(_dev(a)), 1.5, -0.5, N, _p(y))
    ref = 1.5 * _f(a) - 0.5 * _f(y0)
    _check("vec_axpby", y, ref, F32 * ref.abs() + 2 * U * (1.5 * _f(a).abs() + 0.5 * _f(y0).abs()))
    y = torch.full((N,), math.nan, device=DEV)
    _call("b200_vec_axpby", _p(_dev(a)), 1.5, 0.0, N, _p(y))
    _check("vec_axpby beta 0", y, 1.5 * _f(a), F32 * 1.5 * _f(a).abs())
