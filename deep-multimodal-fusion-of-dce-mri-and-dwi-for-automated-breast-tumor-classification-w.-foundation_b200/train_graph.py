"""Training-mode forward + explicit backward of the encoders on the sm_100a kernels (BASELINE configs C1 / C5).

The reference trains `ModelMaskHeadBackbone` through torch autograd (code/train.py:294-428, code/train_fusion.py:203-321):
train-mode BatchNorm (batch statistics, running-statistics update), active nn.Dropout, every parameter receiving a
gradient.  Here the same arithmetic is an explicit tape:

* every tensor-core convolution = three launches of hand-written kernels - forward `b200_conv_gemm_ex` on the bf16
  packed weights, data gradient `b200_conv_gemm_ex` on the flipped / transposed packing, weight gradient
  `b200_conv_wgrad` (tcgen05 with MN-major operands straight from the NHWC maps; csrc/conv_wgrad.cu);
* BatchNorm statistics / apply / backward, activations, residual adds, dropout (Philox, regenerated in the backward
  pass), squeeze-excite, the mask head and mask-guided attention, the 1-channel convolutions, the stem, the
  classifier and every loss term are the SIMT kernels of csrc/train_elem.cu;
* PyTorch provides device memory, the parameter objects and (optionally) torch.distributed - no ATen arithmetic on
  maps, no autograd engine.

Activations and their gradients are NHWC bf16, parameter gradients fp32 accumulated straight into `param.grad` in the
parameter's own layout, BatchNorm buffers updated in place like nn.BatchNorm2d does.  Covers the CNN encoder
configuration of BASELINE.json (block1 reading the raw <= 32-channel input with stride 2, stride-1 block2 / block3,
one bottleneck per block, mask head on f2): anything else raises.
"""
from __future__ import annotations

import torch
import torch.nn as nn

import b200_native as nat

_P = nat._ptr


def _s():
    return nat._stream()


def _call(name, *args):
    nat._call(name, None, *args)


class Tape:
    """Reverse-mode bookkeeping: `grads` maps a tensor's id to the gradient accumulated so far (bf16 maps / fp32
    vectors); `steps` are closures run in reverse order by `backward`."""

    def __init__(self):
        self.steps = []
        self.grads = {}
        self.keep = []  # tensors referenced by id must stay alive

    def record(self, fn):
        self.steps.append(fn)

    def grad_of(self, t):
        return self.grads.pop(id(t), None)

    def add_grad(self, t, g):
        """Accumulate gradient g for tensor t (takes ownership of g on first use)."""
        self.keep.append(t)
        cur = self.grads.get(id(t))
        if cur is None:
            self.grads[id(t)] = g
        elif g.dtype == torch.bfloat16:
            C = g.shape[-1]
            _call("b200_map_axpby", _P(cur), nat._ld(cur), 1.0, _P(g), nat._ld(g), 1.0, g.numel() // C, C, _P(cur),
                  nat._ld(cur), _s())
        else:
            _call("b200_vec_axpby", _P(g), 1.0, 1.0, g.numel(), _P(cur), _s())

    def backward(self, want=()):
        """Run the recorded steps in reverse.  `want`: input tensors whose accumulated gradient is returned (None where
        nothing reached them)."""
        for fn in reversed(self.steps):
            fn()
        out = [self.grads.get(id(t)) for t in want]
        self.steps.clear()
        self.grads.clear()
        self.keep.clear()
        return out


def _grad_buf(p):
    if p.grad is None:
        p.grad = torch.zeros_like(p, dtype=torch.float32)
    return p.grad


def _rows(t):
    return t.numel() // t.shape[-1]


class _Scratch:
    """Reusable device scratch (fp64 reduction buffers)."""

    def __init__(self, dev):
        self.d2c = torch.zeros(2 * 2048, dtype=torch.float64, device=dev)


# ------------------------------------------------------------------------------------------------------------------
# differentiable building blocks
# ------------------------------------------------------------------------------------------------------------------
class TrainOps:
    def __init__(self, dev, drop_seed=0x5EED):
        self.dev = dev
        self.tape = Tape()
        self.scratch = _Scratch(dev)
        self._packs = {}
        self._bucket_marks = None
        self._seed = int(drop_seed)
        self._launch = 0

    def next_seed(self):
        self._launch += 1
        return (self._seed * 0x9E3779B97F4A7C15 + self._launch * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF

    # ---- weights ------------------------------------------------------------------------------------------------
    def packed(self, conv, need_dgrad=True):
        """bf16 operands of a tensor-core conv, repacked from the fp32 master weights (once per step)."""
        key = id(conv)
        if key in self._packs:
            return self._packs[key]
        w = conv.weight
        cout, cin, kh, kw = w.shape
        taps = kh * kw
        if taps not in (1, 9) or conv.stride != (1, 1) or cin % 64 or cout % 64:
            raise NotImplementedError(f"training path: conv {tuple(w.shape)} stride {conv.stride}")
        wf = torch.empty((cout, taps * cin), dtype=torch.bfloat16, device=self.dev)
        wd = torch.empty((cin, taps * cout), dtype=torch.bfloat16, device=self.dev) if need_dgrad else None
        _call("b200_pack_conv_weights", _P(w.detach()), cout, cin, taps, _P(wf), _P(wd), _s())
        self._packs[key] = (wf, wd, taps)
        return self._packs[key]

    def new_step(self):
        self._packs.clear()

    # ---- convolution (tensor cores) -------------------------------------------------------------------------------
    def conv(self, x, conv, x_needs_grad=True):
        """z = conv(x) without bias (the bias, if any, is applied by bn_act as `beta`).  x NHWC bf16."""
        wf, wd, taps = self.packed(conv, x_needs_grad)
        z = nat.conv_gemm(x, wf, taps=taps)
        tape = self.tape

        def bwd():
            dz = tape.grad_of(z)
            if dz is None:
                return
            B, H, W, cin = x.shape
            cout = z.shape[-1]
            if conv.weight.requires_grad:
                _call("b200_conv_wgrad", _P(dz), nat._ld(dz), _P(x), nat._ld(x), _P(_grad_buf(conv.weight)), B, H, W, cin,
                      cout, taps, _s())
            if x_needs_grad:
                tape.add_grad(x, nat.conv_gemm(dz, wd, taps=taps))

        tape.record(bwd)
        return z

    # ---- BatchNorm (batch statistics) + residual + activation + dropout ---------------------------------------------
    def bn_act(self, z, bn=None, bias=None, act=0, res=None, drop_p=0.0, train_bn=True):
        """a = dropout(act(BN(z) + res)); `bn` an nn.BatchNorm2d in training mode (or None: `bias` only)."""
        R, C = _rows(z), z.shape[-1]
        dev = self.dev
        mean = invstd = gamma = beta = None
        if bn is not None:
            st = self.scratch.d2c[:2 * C]
            st.zero_()
            _call("b200_bn_stats", _P(z), R, C, nat._ld(z), _P(st), _P(st[C:]), _s())
            mean = torch.empty(C, dtype=torch.float32, device=dev)
            invstd = torch.empty(C, dtype=torch.float32, device=dev)
            mom = bn.momentum if bn.momentum is not None else 0.1
            _call("b200_bn_finalize", _P(st), _P(st[C:]), C, float(R), float(bn.eps), float(mom),
                  _P(bn.running_mean) if bn.track_running_stats else None,
                  _P(bn.running_var) if bn.track_running_stats else None, _P(mean), _P(invstd), _s())
            if bn.track_running_stats:
                bn.num_batches_tracked += 1
            gamma, beta = bn.weight, bn.bias
        elif bias is not None:
            beta = bias
        seed = self.next_seed() if drop_p > 0 else 0
        a = torch.empty(z.shape, dtype=torch.bfloat16, device=dev)
        _call("b200_bn_act_fwd", _P(z), nat._ld(z), _P(res), nat._ld(res) if res is not None else 0, _P(mean), _P(invstd),
              _P(gamma.detach()) if gamma is not None else None, _P(beta.detach()) if beta is not None else None, act,
              float(drop_p), seed, R, C, _P(a), nat._ld(a), _s())
        tape = self.tape

        def bwd():
            da = tape.grad_of(a)
            if da is None:
                return
            dz = torch.empty(z.shape, dtype=torch.bfloat16, device=dev)
            dres = torch.empty(res.shape, dtype=torch.bfloat16, device=dev) if res is not None else None
            dg = _grad_buf(gamma) if (gamma is not None and gamma.requires_grad) else None
            db = _grad_buf(beta) if (beta is not None and beta.requires_grad) else None
            _call("b200_bn_act_bwd", _P(z), nat._ld(z), _P(res), nat._ld(res) if res is not None else 0, _P(mean),
                  _P(invstd), _P(gamma.detach()) if gamma is not None else None,
                  _P(beta.detach()) if beta is not None else None, act, float(drop_p), seed, R, C, _P(da), nat._ld(da),
                  1 if bn is not None else 0, _P(self.scratch.d2c), _P(dz), nat._ld(dz), _P(dres),
                  nat._ld(dres) if dres is not None else 0, _P(dg), _P(db), _s())
            tape.add_grad(z, dz)
            if res is not None:
                tape.add_grad(res, dres)

        tape.record(bwd)
        return a

    # ---- squeeze-excite on a map -----------------------------------------------------------------------------------
    def se(self, x, se_mod):
        """SEBlock (reference model_module.py:25-43): returns x * gate, gate."""
        B, H, W, C = x.shape
        npix = H * W
        dev = self.dev
        c1, c2 = se_mod.fc[1], se_mod.fc[3]
        M = c1.out_channels
        sums = torch.empty((B, C), dtype=torch.float32, device=dev)
        _call("b200_map_dot", _P(x), nat._ld(x), None, 0, B, npix, C, _P(sums), _s())
        pooled = torch.empty((B, C), dtype=torch.float32, device=dev)
        gate = torch.empty((B, C), dtype=torch.float32, device=dev)
        _call("b200_se_fwd", _P(sums), B, C, M, npix, _P(c1.weight.detach()), _P(c1.bias.detach()), _P(c2.weight.detach()),
              _P(c2.bias.detach()), _P(pooled), _P(gate), _s())
        y = torch.empty(x.shape, dtype=torch.bfloat16, device=dev)
        _call("b200_map_scale_add", _P(x), nat._ld(x), _P(gate), None, B, npix, C, _P(y), nat._ld(y), 0, _s())
        tape = self.tape

        def bwd():
            dy = tape.grad_of(y)
            if dy is None:
                return
            dgate = torch.empty((B, C), dtype=torch.float32, device=dev)
            _call("b200_map_dot", _P(dy), nat._ld(dy), _P(x), nat._ld(x), B, npix, C, _P(dgate), _s())
            dpooled = torch.empty((B, C), dtype=torch.float32, device=dev)
            da2 = torch.empty((B, C), dtype=torch.float32, device=dev)
            da1 = torch.empty((B, M), dtype=torch.float32, device=dev)
            h = torch.empty((B, M), dtype=torch.float32, device=dev)
            _call("b200_se_bwd", _P(pooled), _P(c1.weight.detach()), _P(c1.bias.detach()), _P(c2.weight.detach()),
                  _P(c2.bias.detach()), _P(dgate), B, C, M, _P(dpooled), _P(da2), _P(da1), _P(h), _s())
            # weight gradients: dW2 [C,M] += da2^T h, dW1 [M,C] += da1^T pooled, biases = column sums
            nat.sgemm(da2, h, _grad_buf(c2.weight).view(C, M), trans_a=True, beta=1)
            nat.sgemm(da1, pooled, _grad_buf(c1.weight).view(M, C), trans_a=True, beta=1)
            nat.colsum(da2, _grad_buf(c2.bias))
            nat.colsum(da1, _grad_buf(c1.bias))
            # dx = dy * gate + dpooled / npix
            _call("b200_vec_axpby", _P(dpooled), 1.0 / npix, 0.0, dpooled.numel(), _P(dpooled), _s())
            dx = torch.empty(x.shape, dtype=torch.bfloat16, device=dev)
            _call("b200_map_scale_add", _P(dy), nat._ld(dy), _P(gate), _P(dpooled), B, npix, C, _P(dx), nat._ld(dx), 0, _s())
            tape.add_grad(x, dx)

        tape.record(bwd)
        return y, gate

    # ---- C -> 1 convolution ---------------------------------------------------------------------------------------------
    def conv_c1(self, x, conv):
        B, H, W, C = x.shape
        taps = conv.kernel_size[0] * conv.kernel_size[1]
        out = torch.empty((B, H, W), dtype=torch.float32, device=self.dev)
        _call("b200_convc1_fwd", _P(x), nat._ld(x), B, H, W, C, taps, _P(conv.weight.detach()),
              _P(conv.bias.detach()) if conv.bias is not None else None, _P(out), _s())
        tape = self.tape

        def bwd():
            do = tape.grad_of(out)
            if do is None:
                return
            dx = torch.empty(x.shape, dtype=torch.bfloat16, device=self.dev)
            _call("b200_convc1_bwd", _P(x), nat._ld(x), _P(do), B, H, W, C, taps, _P(conv.weight.detach()), _P(dx),
                  nat._ld(dx), 0, _P(_grad_buf(conv.weight)), _P(_grad_buf(conv.bias)) if conv.bias is not None else None,
                  _s())
            tape.add_grad(x, dx)

        tape.record(bwd)
        return out

    # ---- 1 -> N convolution of a 1-channel fp32 map ------------------------------------------------------------------------
    def lift(self, r, conv, r_needs_grad=True):
        N = conv.out_channels
        z = torch.empty((*r.shape, N), dtype=torch.bfloat16, device=self.dev)
        _call("b200_lift_fwd", _P(r), r.numel(), N, _P(conv.weight.detach()), _P(z), _s())
        tape = self.tape

        def bwd():
            dz = tape.grad_of(z)
            if dz is None:
                return
            dr = torch.empty(r.shape, dtype=torch.float32, device=self.dev) if r_needs_grad else None
            _call("b200_lift_bwd", _P(dz), _P(r), r.numel(), N, _P(conv.weight.detach()), _P(_grad_buf(conv.weight)), _P(dr),
                  _s())
            if r_needs_grad:
                tape.add_grad(r, dr)

        tape.record(bwd)
        return z

    # ---- map arithmetic -----------------------------------------------------------------------------------------------------
    def add(self, a, b):
        y = nat.add_maps(a, b)
        tape = self.tape

        def bwd():
            dy = tape.grad_of(y)
            if dy is None:
                return
            tape.add_grad(a, dy)
            tape.add_grad(b, _copy_map(dy))

        tape.record(bwd)
        return y

    def mask_modulate(self, f, mask_pred, ma):
        """MaskGuidedSpatialAttention at the map's own size (reference :75-97): returns f * (1 + gamma A), A."""
        B, H, W, C = f.shape
        dev = self.dev
        mp = ma.mask_processor
        K = mp[0].out_channels
        wa, gw, gb, wb, bb = (mp[0].weight, mp[1].weight, mp[1].bias, mp[3].weight, mp[3].bias)
        A = torch.empty((B, H, W), dtype=torch.float32, device=dev)
        nat.mask_attention(mask_pred, (K, wa.detach().flatten(), gw.detach(), gb.detach(), wb.detach().flatten(),
                                       bb.detach(), mp[1].eps), A)
        gamma = ma.gamma.detach().reshape(1)
        y = torch.empty(f.shape, dtype=torch.bfloat16, device=dev)
        nat.scale_map(f, y, attn=A, gamma=gamma)
        tape = self.tape

        def bwd():
            dy = tape.grad_of(y)
            if dy is None:
                return
            df = torch.empty(f.shape, dtype=torch.bfloat16, device=dev)
            dA = torch.empty((B, H, W), dtype=torch.float32, device=dev)
            _call("b200_modulate_bwd", _P(dy), nat._ld(dy), _P(f), nat._ld(f), _P(A), _P(gamma), B * H * W, C, _P(df),
                  nat._ld(df), _P(dA), _P(_grad_buf(ma.gamma)), _s())
            tape.add_grad(f, df)
            dm = torch.empty((B, H, W), dtype=torch.float32, device=dev)
            _call("b200_mask_attn_bwd", _P(mask_pred), _P(dA), B, H * W, K, _P(wa.detach()), _P(gw.detach()),
                  _P(gb.detach()), _P(wb.detach()), _P(bb.detach()), float(mp[1].eps), _P(dm), _P(_grad_buf(wa)),
                  _P(_grad_buf(gw)), _P(_grad_buf(gb)), _P(_grad_buf(wb)), _P(_grad_buf(bb)), _s())
            tape.add_grad(mask_pred, dm)

        tape.record(bwd)
        return y, A


def _copy_map(t):
    out = torch.empty(t.shape, dtype=t.dtype, device=t.device)
    C = t.shape[-1]
    _call("b200_map_axpby", _P(t), nat._ld(t), 1.0, None, 0, 0.0, t.numel() // C, C, _P(out), nat._ld(out), _s())
    return out


# ------------------------------------------------------------------------------------------------------------------
# encoder
# ------------------------------------------------------------------------------------------------------------------
def _check_supported(m):
    if m.use_backbone or m.use_hybrid_transformer:
        raise NotImplementedError("training path: CNN encoders only (no backbone adapter / hybrid transformer stage)")
    if tuple(m.num_repeats) != (1, 1, 1) or m.mask_stage != "f2" or not m.mask_enabled or not m.use_se:
        raise NotImplementedError("training path: repeat_blocks (1,1,1), mask head on f2, squeeze-excite on")
    if m.block1.stride != 2 or m.block2.stride != 1 or m.block3.stride != 1:
        raise NotImplementedError("training path: downsample=(True, False, False)")
    if m.modality_attention is None:
        raise NotImplementedError("training path: modality attention on")


def _block_tail(ops, blk, t2, identity, p_drop):
    """conv 1x1 -> BN, + identity, GELU, Dropout, SE, ReconHead (reference :298-316)."""
    bt = blk.bottlenecks[0]
    z3 = ops.conv(t2, bt[7])
    out = ops.bn_act(z3, bn=bt[8], act=1, res=identity, drop_p=p_drop)
    out, _ = ops.se(out, blk.se)
    rec = None
    if blk.reconstruct is not None:
        rh = blk.reconstruct.conv
        ar = ops.bn_act(ops.conv(out, rh[0]), bn=rh[1], act=1)
        rec = ops.conv_c1(ar, rh[3])
    return out, rec


def _block_from_map(ops, blk, x, p_drop):
    bt = blk.bottlenecks[0]
    identity = ops.bn_act(ops.conv(x, blk.skip[0]), bn=blk.skip[1]) if blk.skip is not None else x
    t1 = ops.bn_act(ops.conv(x, bt[0]), bn=bt[1], act=1, drop_p=p_drop)
    t2 = ops.bn_act(ops.conv(t1, bt[4]), bn=bt[5], act=1)
    return _block_tail(ops, blk, t2, identity, p_drop)


def _projector(ops, pr, src):
    g = ops.bn_act(ops.conv(src, pr.proj[0]), bn=pr.proj[1], act=1)
    return ops.bn_act(ops.conv(g, pr.proj[3]), bn=pr.proj[4], act=1)


def _projector_c1(ops, pr, r):
    g = ops.bn_act(ops.lift(r, pr.proj[0], r_needs_grad=False), bn=pr.proj[1], act=1)
    return ops.bn_act(ops.conv(g, pr.proj[3]), bn=pr.proj[4], act=1)


def encoder_forward_train(ops, m, x, heads=True):
    """Train-mode ModelMaskHeadBackbone.forward (reference :645-733) on the tape of `ops`.

    x [B,C,H,W] fp32 normalised input.  Returns a dict: logits [B,K] fp32, f1 / f2 / f3 NHWC bf16, r1 / r2 fp32
    [B,h,w], p1 / p1_r / p2 / p2_r NHWC bf16 at the MAP resolution (the reference's AdaptiveAvgPool2d to 2x the size
    replicates every pixel 2 x 2, which changes neither the BatchNorm statistics nor the cosine / mean losses taken on
    the result), mask_pred [B,h,w] fp32, mask_attn_map, mod_attn_map, pooled3 (the classifier's GAP input).
    heads=False skips the encoder's own classifier and projectors (the fusion step's loss does not read them, so the
    reference's autograd leaves their parameters without a gradient too)."""
    _check_supported(m)
    dev = x.device
    tape = ops.tape
    x = x.contiguous().float()
    B, C, H, W = x.shape
    p_drop = float(m.dropout)
    b1 = m.block1
    stride = b1.stride
    Ho, Wo = H // stride, W // stride
    marks = getattr(ops, "_bucket_marks", None) or [None, None, None]
    if marks[0] is not None:
        tape.record(marks[0])
    # ---- modality attention + the two strided 1x1 convolutions that read the raw input (fp32 SIMT "stem") ----
    se0 = m.modality_attention
    pm = torch.empty(B * C, dtype=torch.float32, device=dev)
    nat.plane_mean(x, B * C, H * W, pm)
    skip_conv, mid_conv = b1.skip[0], b1.bottlenecks[0][0]
    n_skip, n_mid = skip_conv.out_channels, mid_conv.out_channels
    n_cat = n_skip + n_mid
    wcat = torch.cat([skip_conv.weight.detach().flatten(1), mid_conv.weight.detach().flatten(1)], 0).contiguous()
    ones = torch.ones(n_cat, dtype=torch.float32, device=dev)
    zeros = torch.zeros(n_cat, dtype=torch.float32, device=dev)
    zcat = torch.empty((B, Ho, Wo, n_cat), dtype=torch.bfloat16, device=dev)
    dummy = torch.empty(8, dtype=torch.bfloat16, device=dev)
    gate0 = torch.empty((B, C), dtype=torch.float32, device=dev)
    c1, c2 = se0.fc[1], se0.fc[3]
    nat.stem(x, stride, pm, (c1.weight.detach().flatten(1), c1.bias.detach(), c2.weight.detach().flatten(1), c2.bias.detach()),
             wcat, ones, zeros, n_cat, 0, zcat, dummy, gate0)
    z_skip, z_mid = zcat[..., :n_skip], zcat[..., n_skip:]

    def stem_bwd():
        dzs, dzm = tape.grad_of(z_skip), tape.grad_of(z_mid)
        if dzs is None and dzm is None:
            return
        dz = torch.zeros((B, Ho, Wo, n_cat), dtype=torch.bfloat16, device=dev)
        for part, g in ((dz[..., :n_skip], dzs), (dz[..., n_skip:], dzm)):
            if g is not None:
                _call("b200_map_axpby", _P(g), nat._ld(g), 1.0, None, 0, 0.0, _rows(g), g.shape[-1], _P(part), n_cat, _s())
        dw = torch.zeros((n_cat, C), dtype=torch.float32, device=dev)
        dgate = torch.zeros((B, C), dtype=torch.float32, device=dev)
        _call("b200_stem_bwd", _P(x), B, C, H, W, stride, _P(gate0), _P(dz), n_cat, _P(wcat), _P(dw), _P(dgate), _s())
        _call("b200_vec_axpby", _P(dw[:n_skip]), 1.0, 1.0, n_skip * C, _P(_grad_buf(skip_conv.weight)), _s())
        _call("b200_vec_axpby", _P(dw[n_skip:]), 1.0, 1.0, n_mid * C, _P(_grad_buf(mid_conv.weight)), _s())
        # modality SE: gate = sigmoid(W2 gelu(W1 pm + b1) + b2) with pm the plane means
        M = c1.out_channels
        dpooled = torch.empty((B, C), dtype=torch.float32, device=dev)
        da2 = torch.empty((B, C), dtype=torch.float32, device=dev)
        da1 = torch.empty((B, M), dtype=torch.float32, device=dev)
        h = torch.empty((B, M), dtype=torch.float32, device=dev)
        pooled = pm.view(B, C)
        _call("b200_se_bwd", _P(pooled), _P(c1.weight.detach()), _P(c1.bias.detach()), _P(c2.weight.detach()),
              _P(c2.bias.detach()), _P(dgate), B, C, M, _P(dpooled), _P(da2), _P(da1), _P(h), _s())
        nat.sgemm(da2, h, _grad_buf(c2.weight).view(C, M), trans_a=True, beta=1)
        nat.sgemm(da1, pooled, _grad_buf(c1.weight).view(M, C), trans_a=True, beta=1)
        nat.colsum(da2, _grad_buf(c2.bias))
        nat.colsum(da1, _grad_buf(c1.bias))

    tape.record(stem_bwd)
    bt1 = b1.bottlenecks[0]
    identity1 = ops.bn_act(z_skip, bn=b1.skip[1])
    t1 = ops.bn_act(z_mid, bn=bt1[1], act=1, drop_p=p_drop)
    t2 = ops.bn_act(ops.conv(t1, bt1[4]), bn=bt1[5], act=1)
    f1, r1 = _block_tail(ops, b1, t2, identity1, p_drop)
    # ---- block2, mask head on f2 (+ aligned f1), mask-guided modulation -------------------------------------------
    if marks[1] is not None:
        tape.record(marks[1])
    f2_pre, r2 = _block_from_map(ops, m.block2, f1, p_drop)
    al = m.f1_to_f2.proj
    if isinstance(al, nn.Identity):
        f1_aligned = f1
    else:
        f1_aligned = ops.bn_act(ops.conv(f1, al[0]), bn=al[1], act=1)
    m_in = ops.add(f2_pre, f1_aligned)
    mh = m.mask_head
    if m_in.shape[1] != m.mask_size:
        raise NotImplementedError("training path: mask head at the mask size (32 x 32 maps)")
    t64 = ops.bn_act(ops.conv(m_in, mh.pre), bias=mh.pre.bias)
    mask_pred = ops.conv_c1(t64, mh.out)
    f2, attn_map = ops.mask_modulate(f2_pre, mask_pred, m.mask_spatial_attention)
    # ---- block3, classifier, projectors ------------------------------------------------------------------------------
    if marks[2] is not None:
        tape.record(marks[2])
    f3, _ = _block_from_map(ops, m.block3, f2, p_drop)
    logits = pooled3 = p1 = p2 = p1_r = p2_r = None
    if heads:
        npix3 = f3.shape[1] * f3.shape[2]
        C3 = f3.shape[-1]
        sums3 = torch.empty((B, C3), dtype=torch.float32, device=dev)
        _call("b200_map_dot", _P(f3), nat._ld(f3), None, 0, B, npix3, C3, _P(sums3), _s())
        head = m.classification_head
        K = head.fc.out_features
        logits = torch.empty((B, K), dtype=torch.float32, device=dev)
        pooled3 = torch.empty((B, C3), dtype=torch.float32, device=dev)
        _call("b200_vec_axpby", _P(sums3), 1.0 / npix3, 0.0, sums3.numel(), _P(pooled3), _s())  # GAP mean (pre-normalise)
        nat.cls_head(sums3, None, npix3, head.fc.weight.detach(), head.fc.bias.detach(), head.normalize, logits)

        def head_bwd():
            dl = tape.grad_of(logits)
            if dl is None:
                return
            dpooled = torch.empty((B, C3), dtype=torch.float32, device=dev)
            _call("b200_cls_head_bwd", _P(pooled3), _P(dl), _P(head.fc.weight.detach()), B, C3, K, 1 if head.normalize else 0,
                  _P(_grad_buf(head.fc.weight)), _P(_grad_buf(head.fc.bias)), _P(dpooled), _s())
            _call("b200_vec_axpby", _P(dpooled), 1.0 / npix3, 0.0, dpooled.numel(), _P(dpooled), _s())
            df3 = torch.empty(f3.shape, dtype=torch.bfloat16, device=dev)
            _call("b200_map_scale_add", None, 0, None, _P(dpooled), B, npix3, C3, _P(df3), nat._ld(df3), 0, _s())  # broadcast
            tape.add_grad(f3, df3)

        tape.record(head_bwd)
        p1 = _projector(ops, m.proj_f1, f1)
        p2 = _projector(ops, m.proj_f2, f2)
        p1_r = _projector_c1(ops, m.proj_r1, r1)
        p2_r = _projector_c1(ops, m.proj_r2, r2)
    return {"logits": logits, "f1": f1, "f2": f2, "f3": f3, "r1": r1, "r2": r2, "p1": p1, "p1_r": p1_r, "p2": p2,
            "p2_r": p2_r, "mask_pred": mask_pred, "mask_attn_map": attn_map, "mod_attn_map": gate0, "pooled3": pooled3,
            "x": x}


# ------------------------------------------------------------------------------------------------------------------
# the single-modality objective (BASELINE config C1): LightningSingleModel._shared_step, code/train.py:294-400
# ------------------------------------------------------------------------------------------------------------------
def single_model_loss(ops, out, masks, labels, *, smoothing, gamma, class_weights, lambda_mask, lambda_recon,
                      lambda_mimic, lambda_feat_norm, aux_w=1.0):
    """Seeds the tape with the gradients of
        cls + lambda_feat_norm * sum_f mean(f^2) + lambda_mask * dice + lambda_recon * (recon * lambda_recon * aux_w) * aux_w
            + lambda_mimic * (mimic * lambda_mimic * aux_w) * aux_w
    (the reference weights the last two twice, train.py:396-399 and :462-464 - reproduced) and returns
    (total [1] fp32 device tensor, parts dict of device scalars)."""
    tape, dev = ops.tape, ops.dev
    logits = out["logits"]
    B, K = logits.shape
    parts = {k: torch.zeros(1, dtype=torch.float32, device=dev) for k in ("cls", "feat_norm", "mask", "recon", "mimic")}
    dl = torch.empty_like(logits)
    cw = class_weights.to(dev).float().contiguous() if class_weights is not None else None
    _call("b200_focal_loss", _P(logits), _P(labels), B, K, float(smoothing), float(gamma), _P(cw), 1.0 / B, _P(parts["cls"]),
          _P(dl), _s())
    tape.add_grad(logits, dl)
    # feature-norm regulariser: sum_f mean(f^2), gradient 2 f / numel
    fn64 = torch.zeros(3, dtype=torch.float64, device=dev)
    for i, key in enumerate(("f1", "f2", "f3")):
        f = out[key]
        C = f.shape[-1]
        _call("b200_map_sumsq", _P(f), nat._ld(f), _rows(f), C, _P(fn64[i:]), _s())
        if lambda_feat_norm != 0:
            g = torch.empty(f.shape, dtype=torch.bfloat16, device=dev)
            _call("b200_map_axpby", _P(f), nat._ld(f), 2.0 * lambda_feat_norm / f.numel(), None, 0, 0.0, _rows(f), C, _P(g),
                  nat._ld(g), _s())
            tape.add_grad(f, g)
    numels = torch.tensor([out[k].numel() for k in ("f1", "f2", "f3")], dtype=torch.float64, device=dev)
    parts["feat_norm"] = (fn64 / numels).sum().float().reshape(1)
    # mask dice
    mp = out["mask_pred"]
    n = mp[0].numel()
    dm = torch.empty_like(mp)
    _call("b200_dice_loss", _P(mp), _P(masks.contiguous().float()), B, n, 1e-6, 1.0 / B, _P(parts["mask"]), _P(dm), _s())
    _call("b200_vec_axpby", _P(dm), float(lambda_mask), 0.0, dm.numel(), _P(dm), _s())
    tape.add_grad(mp, dm)
    # reconstruction (both heads) and mimic (both pairs)
    x = out["x"]
    _, C, H, W = x.shape
    w_recon = lambda_recon * lambda_recon * aux_w * aux_w
    for key in ("r1", "r2"):
        r = out[key]
        dr = torch.empty_like(r)
        one = torch.zeros(1, dtype=torch.float32, device=dev)
        _call("b200_recon_loss", _P(r), B, r.shape[1], r.shape[2], _P(x), C, None, 0, H, W, 1e-3, 1.0 / (B * H * W), _P(one), _P(dr), _s())
        _call("b200_vec_axpby", _P(one), 1.0, 1.0, 1, _P(parts["recon"]), _s())
        _call("b200_vec_axpby", _P(dr), float(w_recon), 0.0, dr.numel(), _P(dr), _s())
        tape.add_grad(r, dr)
    w_mimic = lambda_mimic * lambda_mimic * aux_w * aux_w
    for s_key, t_key in (("p1", "p1_r"), ("p2", "p2_r")):
        s_map, t_map = out[s_key], out[t_key]
        ds = torch.empty(s_map.shape, dtype=torch.bfloat16, device=dev)
        _call("b200_mimic_loss", _P(s_map), _P(t_map), B, s_map[0].numel(), float(w_mimic) / B, _P(parts["mimic"]), _P(ds), _s())
        tape.add_grad(s_map, ds)
    if w_mimic != 0:
        parts["mimic"] = parts["mimic"] / w_mimic
    total = (parts["cls"] + lambda_feat_norm * parts["feat_norm"] + lambda_mask * parts["mask"] +
             w_recon * parts["recon"] + w_mimic * parts["mimic"])
    return total, parts


# ------------------------------------------------------------------------------------------------------------------
# fusion head at full resolution (reference model_module.py:919-1000, train mode)
# ------------------------------------------------------------------------------------------------------------------
def _split_k(m, n, k):
    tiles = ((m + 63) // 64) * ((n + 63) // 64)
    return max(1, min((2 * 148 + tiles - 1) // tiles, max(1, k // 64)))


def _wgrad32(dy, x, param, rows=None):
    """param.grad[rows] += dy^T x (fp32 token / vector matrices)."""
    g = _grad_buf(param) if rows is None else _grad_buf(param)[rows]
    g = g.view(g.shape[0], -1)
    nat.sgemm(dy, x, g, trans_a=True, beta=1, split_k=_split_k(g.shape[0], g.shape[1], dy.shape[0]))


def _bgrad32(dy, param, rows=None):
    nat.colsum(dy, _grad_buf(param) if rows is None else _grad_buf(param)[rows])


def fusion_forward_train(ops, fm, f3d, f3c, md, mc):
    """Train-mode FusionModel.forward on the tape of `ops`.  f3d / f3c: NHWC bf16 encoder maps (tape tensors when the
    encoders train too), md / mc: [B,h,w] fp32 encoder mask logits (or None without use_mask_attention).  The
    reference's dead cat -> reduce -> refine branch (:935-940) is not evaluated.  Returns a dict: logits, fused_mask
    [B,h,w] fp32, recon [B,h,w] fp32, proj NHWC bf16, gating [B,2], attn_weights, p_dwi, p_dce."""
    from model_module import _bilinear_axis_weights

    if isinstance(fm.proj_in_dwi, nn.Identity) or isinstance(fm.proj_in_dce, nn.Identity) or fm.fusion_se is None:
        raise NotImplementedError("training path: proj_in convolutions and fusion_se present")
    if not fm.use_cross_attention:
        raise NotImplementedError("training path: use_cross_attention")
    tape, dev = ops.tape, ops.dev
    B, H, W, _ = f3d.shape
    C, (hp, wp), NH = fm.fusion_channels, fm.token_pool, fm.mha_heads
    T, npix, R = hp * wp, H * W, B * hp * wp
    if H % hp or W % wp:
        raise NotImplementedError("training path: token bins that tile the map")

    def z(*shape):
        return torch.empty(shape, dtype=torch.float32, device=dev)

    p_d = ops.conv(f3d, fm.proj_in_dwi)
    p_c = ops.conv(f3c, fm.proj_in_dce)
    sum_d, sum_c = z(B, C), z(B, C)
    _call("b200_map_dot", _P(p_d), nat._ld(p_d), None, 0, B, npix, C, _P(sum_d), _s())
    _call("b200_map_dot", _P(p_c), nat._ld(p_c), None, 0, B, npix, C, _P(sum_c), _s())
    Td, Tc = z(R, C), z(R, C)
    nat.fusion_tokens(p_d, hp, wp, Td.view(B, T, C))
    nat.fusion_tokens(p_c, hp, wp, Tc.view(B, T, C))
    # ---- cross-attention block on the pooled tokens (fp32) ----
    ca = fm.cross_attn_block
    Win, b_in = ca.cross_attn.in_proj_weight.detach(), ca.cross_attn.in_proj_bias.detach()
    Wo, bo = ca.cross_attn.out_proj.weight.detach(), ca.cross_attn.out_proj.bias.detach()
    ln = ca.attn_ffn[0]
    W1, b1 = ca.attn_ffn[1].weight.detach(), ca.attn_ffn[1].bias.detach()
    W2, b2 = ca.attn_ffn[3].weight.detach(), ca.attn_ffn[3].bias.detach()
    Q, KV, Pm, CTX, AO, LN = z(R, C), z(R, 2 * C), z(B, NH, T, T), z(R, C), z(R, C), z(R, C)
    mean, rstd, H1, G1, LOW = z(R), z(R), z(R, C), z(R, C), z(R, C)
    nat.sgemm(Td, Win[:C], Q, trans_b=True, bias=b_in[:C])
    nat.sgemm(Tc, Win[C:], KV, trans_b=True, bias=b_in[C:])
    Kt, Vt = KV[:, :C], KV[:, C:]
    nat.mha_fwd(Q, Kt, Vt, B, NH, Pm, CTX)
    nat.sgemm(CTX, Wo, AO, trans_b=True, bias=bo)
    nat.ln_fwd(AO, ln.weight.detach(), ln.bias.detach(), ln.eps, LN, mean, rstd)
    nat.sgemm(LN, W1, G1, trans_b=True, bias=b1, pre=H1, act=1)
    nat.sgemm(G1, W2, LOW, trans_b=True, bias=b2, res=AO)
    # ---- gating ----
    use_ma = bool(fm.use_mask_attention)
    if use_ma and (md is None or mc is None):
        raise RuntimeError("use_mask_attention needs both encoder mask predictions")
    D = 2 * C + (2 if use_ma else 0)
    gx, alpha = z(B, D), z(B, 2)
    npm = md[0].numel() if use_ma else 0
    gw, gb = fm.gating.fc.weight, fm.gating.fc.bias
    _call("b200_gating_fwd", _P(sum_d), _P(sum_c), B, C, npix, _P(md) if use_ma else None, _P(mc) if use_ma else None, npm,
          _P(gw.detach()), _P(gb.detach()), _P(gx), _P(alpha), _s())
    # ---- fused = alpha0 p_dwi + alpha1 p_dce + up(lowres) ----
    fused = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=dev)
    nat.fusion_mix(p_d, p_c, alpha, LOW.view(B, T, C), None, hp, wp, fused)
    attn_w = None  # (the head-averaged attention weights are an eval-path output; training does not need them)

    def mix_bwd():
        df = tape.grad_of(fused)
        if df is None:
            return
        dalpha = torch.zeros((B, 2), dtype=torch.float32, device=dev)
        dLOW = torch.zeros((R, C), dtype=torch.float32, device=dev)
        _call("b200_fusion_mix_bwd", _P(df), _P(p_d), _P(p_c), None, B, H, W, C, hp, wp, _P(dalpha), _P(dLOW), None, None,
              None, None, None, None, 0, _s())
        # cross-attention block backward (same sequence as the fusion-head trainer, csrc/train_ops.cu kernels)
        dG1, dH1, dLN, dAO, tmp, dCTX, dQ, dKV = z(R, C), z(R, C), z(R, C), z(R, C), z(R, C), z(R, C), z(R, C), z(R, 2 * C)
        _wgrad32(dLOW, G1, ca.attn_ffn[3].weight)
        _bgrad32(dLOW, ca.attn_ffn[3].bias)
        nat.sgemm(dLOW, W2, dG1)
        nat.gelu_bwd(H1, dG1, dH1)
        _wgrad32(dH1, LN, ca.attn_ffn[1].weight)
        _bgrad32(dH1, ca.attn_ffn[1].bias)
        nat.sgemm(dH1, W1, dLN)
        nat.ln_bwd(AO, dLN, dLOW, ln.weight.detach(), mean, rstd, dAO, tmp)
        _bgrad32(tmp, ln.weight)
        _bgrad32(dLN, ln.bias)
        _wgrad32(dAO, CTX, ca.cross_attn.out_proj.weight)
        _bgrad32(dAO, ca.cross_attn.out_proj.bias)
        nat.sgemm(dAO, Wo, dCTX)
        nat.mha_bwd(Q, Kt, Vt, Pm, dCTX, B, NH, dQ, dKV[:, :C], dKV[:, C:])
        _wgrad32(dQ, Td, ca.cross_attn.in_proj_weight, slice(0, C))
        _bgrad32(dQ, ca.cross_attn.in_proj_bias, slice(0, C))
        _wgrad32(dKV, Tc, ca.cross_attn.in_proj_weight, slice(C, 3 * C))
        _bgrad32(dKV, ca.cross_attn.in_proj_bias, slice(C, 3 * C))
        dTd, dTc = z(R, C), z(R, C)
        nat.sgemm(dQ, Win[:C], dTd)
        nat.sgemm(dKV, Win[C:], dTc)
        bin_px = (H // hp) * (W // wp)
        _call("b200_vec_axpby", _P(dTd), 1.0 / bin_px, 0.0, dTd.numel(), _P(dTd), _s())
        _call("b200_vec_axpby", _P(dTc), 1.0 / bin_px, 0.0, dTc.numel(), _P(dTc), _s())
        # gating backward
        dgl, dgx, dpv_d, dpv_c = z(B, 2), z(B, D), z(B, C), z(B, C)
        _call("b200_gating_bwd", _P(alpha), _P(dalpha), _P(gw.detach()), B, C, D, npix, _P(dgl), _P(dgx), _P(dpv_d),
              _P(dpv_c), _s())
        _wgrad32(dgl, gx, gw)
        _bgrad32(dgl, gb)
        if use_ma:
            for m_, col in ((md, 2 * C), (mc, 2 * C + 1)):
                dm_ = torch.empty(m_.shape, dtype=torch.float32, device=dev)
                _call("b200_row_bcast", _P(dgx[:, col:]), D, 1.0 / npm, B, npm, _P(dm_), _s())
                tape.add_grad(m_, dm_)
        dpd = torch.empty(p_d.shape, dtype=torch.bfloat16, device=dev)
        dpc = torch.empty(p_c.shape, dtype=torch.bfloat16, device=dev)
        _call("b200_fusion_mix_bwd", _P(df), None, None, _P(alpha), B, H, W, C, hp, wp, None, None, _P(dTd), _P(dTc),
              _P(dpv_d), _P(dpv_c), _P(dpd), _P(dpc), 1, _s())
        tape.add_grad(p_d, dpd)
        tape.add_grad(p_c, dpc)

    tape.record(mix_bwd)
    fr, gate = ops.se(fused, fm.fusion_se)
    # ---- heads on fused_refined ----
    mh = fm.mask_head
    if H != fm.mask_size:
        raise NotImplementedError("training path: mask head at the mask size (32 x 32 maps)")
    t64 = ops.bn_act(ops.conv(fr, mh.pre), bias=mh.pre.bias)
    fused_mask = ops.conv_c1(t64, mh.out)
    sums = z(B, C)
    _call("b200_map_dot", _P(fr), nat._ld(fr), None, 0, B, npix, C, _P(sums), _s())
    pooled = z(B, C)
    _call("b200_vec_axpby", _P(sums), 1.0 / npix, 0.0, sums.numel(), _P(pooled), _s())
    fc = fm.classifier[2]
    K = fc.out_features
    logits = z(B, K)
    nat.cls_head(sums, None, npix, fc.weight.detach(), fc.bias.detach(), False, logits)

    def cls_bwd():
        dl = tape.grad_of(logits)
        if dl is None:
            return
        dpooled = z(B, C)
        _call("b200_cls_head_bwd", _P(pooled), _P(dl), _P(fc.weight.detach()), B, C, K, 0, _P(_grad_buf(fc.weight)),
              _P(_grad_buf(fc.bias)), _P(dpooled), _s())
        _call("b200_vec_axpby", _P(dpooled), 1.0 / npix, 0.0, dpooled.numel(), _P(dpooled), _s())
        dfr = torch.empty(fr.shape, dtype=torch.bfloat16, device=dev)
        _call("b200_map_scale_add", None, 0, None, _P(dpooled), B, npix, C, _P(dfr), nat._ld(dfr), 0, _s())
        tape.add_grad(fr, dfr)

    tape.record(cls_bwd)
    rh = fm.fusion_reconstruct.conv
    recon = ops.conv_c1(ops.bn_act(ops.conv(fr, rh[0]), bn=rh[1], act=1), rh[3])
    proj = _projector(ops, fm.projF, fr)
    return {"logits": logits, "fused_mask": fused_mask, "recon": recon, "proj": proj, "gating": alpha, "attn_weights": attn_w,
            "p_dwi": p_d, "p_dce": p_c, "fused_refined": fr}


def fusion_objective(ops, fo, enc_d, enc_c, masks, labels, dwi_in, dce_in, *, smoothing, gamma, class_weights, lambda_mask,
                     lambda_recon, lambda_mimic, aux_w=1.0, md=None, mc=None, frozen_d=None, frozen_c=None):
    """Total loss of LightningFusionModel._shared_step (code/train_fusion.py:238-296) with its gradients seeded on the
    tape:  cls + lambda_mask * (dice(md) + dice(mc) + dice(fused)) / 3
               + lambda_recon * aux_w * (recon_list(dwi) + recon_list(dce) + recon(fused)) / 3
               + lambda_mimic * aux_w * mimic(proj_fused[:4]).
    `fo` = fusion_forward_train's dict; enc_d / enc_c = the encoders' train-forward dicts (their r1 / r2 and mask_pred
    join the loss) or None when the encoders are frozen (then md / mc are the constant mask logits and the encoder
    reconstruction lists count as absent, i.e. 0, as compute_recon_list_loss does).  Returns (total, parts)."""
    tape, dev = ops.tape, ops.dev
    logits = fo["logits"]
    B, K = logits.shape
    parts = {k: torch.zeros(1, dtype=torch.float32, device=dev) for k in ("cls", "mask", "recon", "mimic")}
    dl = torch.empty_like(logits)
    cw = class_weights.to(dev).float().contiguous() if class_weights is not None else None
    _call("b200_focal_loss", _P(logits), _P(labels), B, K, float(smoothing), float(gamma), _P(cw), 1.0 / B, _P(parts["cls"]),
          _P(dl), _s())
    tape.add_grad(logits, dl)
    tgt = masks.contiguous().float()
    md = enc_d["mask_pred"] if enc_d is not None else md
    mc = enc_c["mask_pred"] if enc_c is not None else mc
    for m_, trainable in ((md, enc_d is not None), (mc, enc_c is not None), (fo["fused_mask"], True)):
        n = m_[0].numel()
        dm = torch.empty(m_.shape, dtype=torch.float32, device=dev) if trainable else None
        _call("b200_dice_loss", _P(m_), _P(tgt), B, n, 1e-6, 1.0 / (3 * B), _P(parts["mask"]), _P(dm), _s())
        if trainable and lambda_mask != 0:
            _call("b200_vec_axpby", _P(dm), float(lambda_mask), 0.0, dm.numel(), _P(dm), _s())
            tape.add_grad(m_, dm)
    _, Cd, H, W = dwi_in.shape
    Cc = dce_in.shape[1]
    wr = lambda_recon * aux_w
    scale = 1.0 / (3 * B * H * W)
    for enc, frozen, x in ((enc_d, frozen_d, dwi_in), (enc_c, frozen_c, dce_in)):
        src = enc if enc is not None else frozen
        if src is None or src.get("r1") is None:
            continue  # no reconstruction list: compute_recon_list_loss returns 0
        for key in ("r1", "r2"):  # compute_recon_list_loss: mean over the list's reconstructions
            r = src[key]
            dr = torch.empty_like(r) if enc is not None else None  # (a frozen encoder's term is a constant of the loss)
            _call("b200_recon_loss", _P(r), B, r.shape[1], r.shape[2], _P(x), x.shape[1], None, 0, H, W, 1e-3, 0.5 * scale,
                  _P(parts["recon"]), _P(dr), _s())
            if enc is not None:
                _call("b200_vec_axpby", _P(dr), float(wr), 0.0, dr.numel(), _P(dr), _s())
                tape.add_grad(r, dr)
    r = fo["recon"]
    dr = torch.empty_like(r)
    _call("b200_recon_loss", _P(r), B, r.shape[1], r.shape[2], _P(dwi_in), Cd, _P(dce_in), Cc, H, W, 1e-3, scale,
          _P(parts["recon"]), _P(dr), _s())
    _call("b200_vec_axpby", _P(dr), float(wr), 0.0, dr.numel(), _P(dr), _s())
    tape.add_grad(r, dr)
    proj = fo["proj"]
    if B >= 4:
        wm = lambda_mimic * aux_w
        dpj = torch.empty(proj.shape, dtype=torch.bfloat16, device=dev)
        one = torch.zeros(1, dtype=torch.float32, device=dev)
        _call("b200_mimic_pairs", _P(proj), B, proj.shape[1] * proj.shape[2], proj.shape[3], 1.0, _P(one), None, _s())
        _call("b200_mimic_pairs", _P(proj), B, proj.shape[1] * proj.shape[2], proj.shape[3], float(wm), _P(parts["mimic"]),
              _P(dpj), _s())
        parts["mimic"] = one
        tape.add_grad(proj, dpj)
    total = parts["cls"] + lambda_mask * parts["mask"] + lambda_recon * aux_w * parts["recon"] + lambda_mimic * aux_w * parts["mimic"]
    return total, parts


# ------------------------------------------------------------------------------------------------------------------
# data-parallel training step of the whole model (BASELINE config C5: backbone unfrozen, bf16, NCCL all-reduce)
# ------------------------------------------------------------------------------------------------------------------
_NO_GRAD_PREFIXES_ENC = ("classification_head.", "proj_f1.", "proj_f2.", "proj_r1.", "proj_r2.", "f2_to_f3.", "f2_weight",
                         "f3_weight", "norm_f2.", "norm_f3.", "mask_head.down_")
_NO_GRAD_PREFIXES_FUS = ("fusion_conv_reduce.", "refine.", "mask_head.down_")


class FullFusionTrainer:
    """One optimisation step of LightningFusionModel (code/train_fusion.py:203-321; optimiser
    code/selector_helpers.py:356-742): train-mode forward of the encoders and the fusion head, the full objective,
    explicit backward, bucketed gradient all-reduce overlapped with the rest of the backward pass, one fused AdamW
    launch over the flat parameter buffer.

    The trainable set is what the reference's optimiser would hold: every parameter with requires_grad that the fusion
    objective can reach (the reference's autograd leaves .grad None on the rest and AdamW skips them, SURVEY.md App.
    A-2: encoder classifier / projectors, unused mask-head down-samplers, the dead reduce / refine branch ...).  Frozen
    encoders (`backbone_freeze_on_start`) therefore put the head alone in the buffers; `refresh()` re-binds the buffers
    after a gradual-unfreeze event (selector_helpers.py:523-620), keeping the Adam moments of the parameters that were
    already in and starting the new ones at step 1.  Every trainable parameter is a view of ONE fp32 buffer, its
    gradient a view of a second one; the gradient buffer is cut into buckets in backward order and bucket i's
    all-reduce (NCCL over NVLink) is issued on a side stream as soon as the tape has passed the forward position where
    its last gradient is produced.  `group_fn(name) -> (lr, weight_decay)` gives per-parameter hyper-parameters
    (discriminative learning rates); `encoder_mode` "train" (what Lightning's fit loop does to the frozen encoders too:
    batch-statistic BatchNorm with running-statistics update, active dropout) or "eval" for the frozen phase."""

    def __init__(self, dwi_model, dce_model, fusion_model, *, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=4e-5,
                 smoothing=0.1, gamma=1.5, class_weights=None, lambda_mask=0.2, lambda_recon=0.1, lambda_mimic=0.2,
                 encoders_trainable=None, encoder_mode="train", group_fn=None, process_group=None, bucket_mb=8.0,
                 seed=0x5EED):
        self.dwi, self.dce, self.fusion = dwi_model, dce_model, fusion_model
        self.hp = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.loss_hp = dict(smoothing=smoothing, gamma=gamma, class_weights=class_weights, lambda_mask=lambda_mask,
                            lambda_recon=lambda_recon, lambda_mimic=lambda_mimic)
        if encoders_trainable is False:
            for m in (dwi_model, dce_model):
                if m is not None:
                    for q in m.parameters():
                        q.requires_grad_(False)
        self.encoder_mode = encoder_mode
        self.group_fn = group_fn
        self.group = process_group
        self.step_count = 0
        self.lr_mult = 1.0   # schedulers scale every group's rate through this factor
        self.aux_w = 1.0     # auxiliary-loss weight schedule (train_fusion.py:220-224)
        dev = next(fusion_model.parameters()).device
        if dev.type != "cuda":
            raise nat.B200NativeError("FullFusionTrainer needs the models on a CUDA device (no CPU path)")
        self.dev = dev
        self.ops = TrainOps(dev, drop_seed=seed)
        self.bucket_elems = int(bucket_mb * (1 << 20) / 4)
        self._comm = None
        self._pending = []
        self.flat = None
        self.names = []
        self.refresh()

    # ---- trainable set / flat buffers ---------------------------------------------------------------------------------
    def _segments(self):
        """Trainable parameters in FORWARD order, segment by segment (a segment = one all-reduce bucket unit)."""
        def seg(module, prefixes, names_filter):
            return [(n, p) for n, p in module.named_parameters()
                    if p.requires_grad and not n.startswith(prefixes) and names_filter(n)]

        segments = []
        for tag, m in (("dwi", self.dwi), ("dce", self.dce)):
            if m is None or not any(p.requires_grad for p in m.parameters()):
                segments += [[], [], []]
                continue
            _check_supported(m)
            b1 = lambda n: n.startswith(("modality_attention.", "block1."))
            b2 = lambda n: n.startswith(("block2.", "f1_to_f2.", "mask_head.", "mask_spatial_attention."))
            b3 = lambda n: n.startswith("block3.")
            for filt in (b1, b2, b3):
                segments.append([(f"{tag}.{n}", p) for n, p in seg(m, _NO_GRAD_PREFIXES_ENC, filt)])
        segments.append([(f"fusion.{n}", p) for n, p in seg(self.fusion, _NO_GRAD_PREFIXES_FUS, lambda n: True)])
        return segments

    def refresh(self):
        """(Re)bind the flat buffers to the current trainable set (call after requires_grad flags change)."""
        from fusion_train import flat_size, flat_views

        dev = self.dev
        old = None
        if self.flat is not None:
            old = {n: (m_.clone(), v_.clone(), int(s0.flatten()[0].item()))
                   for n, m_, v_, s0 in zip(self.names, flat_views(self.params, self.flat["m"]),
                                            flat_views(self.params, self.flat["v"]),
                                            flat_views(self.params, self.flat["step0"]))}
            for p_ in self.params:  # detach the old views so that freed parameters keep their values
                p_.data = p_.data.clone()
                p_.grad = None
        self.segments = self._segments()
        named = [np_ for s_ in self.segments for np_ in s_]
        self.names = [n for n, _ in named]
        self.params = [p_ for _, p_ in named]
        self.encoders_trainable = any(n.startswith(("dwi.", "dce.")) for n in self.names)
        n = flat_size(self.params)
        self.flat_numel = n
        self.flat = {k: torch.zeros(n + (1 if k == "g" else 0), dtype=torch.float32, device=dev) for k in ("p", "g", "m", "v", "lr", "wd")}
        self.flat["step0"] = torch.zeros(n, dtype=torch.int32, device=dev)
        views = {k: flat_views(self.params, self.flat[k]) for k in ("p", "g", "m", "v", "lr", "wd", "step0")}
        for i, (name, p_) in enumerate(named):
            views["p"][i].copy_(p_.data.float())
            p_.data = views["p"][i]
            p_.grad = views["g"][i]
            lr_, wd_ = self.group_fn(name) if self.group_fn is not None else (self.hp["lr"], self.hp["weight_decay"])
            views["lr"][i].fill_(float(lr_))
            views["wd"][i].fill_(float(wd_))
            if old is not None and name in old and old[name][0].shape == views["m"][i].shape:
                views["m"][i].copy_(old[name][0])
                views["v"][i].copy_(old[name][1])
                views["step0"][i].fill_(old[name][2])
            else:
                views["step0"][i].fill_(self.step_count)  # a parameter that joins now counts its Adam steps from here
        ends, off = [], 0
        for s_ in self.segments:
            off += flat_size([p_ for _, p_ in s_])
            ends.append(off)
        self.seg_ends = ends
        self.numel = sum(p_.numel() for p_ in self.params)

    # ---- gradient exchange ---------------------------------------------------------------------------------------------
    def _world(self):
        import torch.distributed as dist

        return dist.get_world_size(self.group) if (dist.is_available() and dist.is_initialized()) else 1

    def _reduce_range(self, lo, hi):
        """SUM all-reduce of flat_g[lo:hi] on the communication stream, ordered after everything recorded so far on the
        compute stream."""
        import torch.distributed as dist

        if self._world() == 1 or hi <= lo:
            return
        if torch.device(self.dev).type != "cuda":  # host-side tests of the bucket plan (gloo): no streams to order
            dist.all_reduce(self.flat["g"][lo:hi], op=dist.ReduceOp.SUM, group=self.group)
            return
        if self._comm is None:
            self._comm = torch.cuda.Stream(device=self.dev)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self._comm):
            self._comm.wait_event(ev)
            self._pending.append(dist.all_reduce(self.flat["g"][lo:hi], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def _marker(self, seg_index):
        """Tape step recorded BEFORE segment seg_index's forward: in the backward pass it runs right after that
        segment's last gradient has been produced, i.e. gradients [seg start, end of buffer) are final."""
        def fire():
            lo = self.seg_ends[seg_index - 1] if seg_index > 0 else 0
            hi = self._reduced_from
            if hi - lo >= self.bucket_elems or seg_index == 0:
                self._reduce_range(lo, hi)
                self._reduced_from = lo
        return fire

    # ---- the step ----------------------------------------------------------------------------------------------------------
    def zero_grad(self):
        self.flat["g"].zero_()

    def _frozen_encoder_outputs(self, m, x):
        """f3 (NHWC bf16) and mask logits [B,h,w] of a frozen encoder: its train-mode forward (batch statistics, dropout,
        running statistics updated - what the reference's fit loop does to frozen encoders) with the tape discarded, or
        its eval forward."""
        if self.encoder_mode == "train":
            ops = TrainOps(self.dev, drop_seed=self.ops.next_seed())
            out = encoder_forward_train(ops, m, x, heads=False)
            ops.tape.steps.clear()
            return out["f3"], out["mask_pred"], out["r1"], out["r2"]
        was = m.training
        m.eval()
        try:
            with torch.no_grad():
                o = m(x, None)
        finally:
            m.train(was)
        rf = o[1].get("recon_feats") or [None, None]
        r1, r2 = (r[:, 0].contiguous() if r is not None else None for r in rf)
        return o[1]["raw_feats"][-1].permute(0, 2, 3, 1), o[2][:, 0].contiguous(), r1, r2

    def forward_backward(self, dwi_in, dce_in, masks, labels, md=None, mc=None, f3d=None, f3c=None):
        """Forward + loss + backward on one batch (gradients ACCUMULATE into the flat buffer: call zero_grad first).
        dwi_in / dce_in: normalised fp32 [B,C,H,W].  Pre-computed frozen-encoder outputs may be passed as f3d / f3c
        (NHWC bf16) and md / mc.  Returns (total, parts)."""
        ops = self.ops
        ops.new_step()
        self._reduced_from = self.flat_numel
        self._pending = []
        labels = labels.to(self.dev, torch.int64).contiguous()
        masks = masks.to(self.dev).float().contiguous()
        enc_d = enc_c = None
        trainable = {"dwi": any(n.startswith("dwi.") for n in self.names), "dce": any(n.startswith("dce.") for n in self.names)}
        outs = {}
        for si, (tag, m, x, pre) in enumerate((("dwi", self.dwi, dwi_in, (f3d, md)), ("dce", self.dce, dce_in, (f3c, mc)))):
            if trainable[tag]:
                marks = [self._marker(3 * si), self._marker(3 * si + 1), self._marker(3 * si + 2)]
                outs[tag] = _encoder_with_markers(ops, m, x, marks)
            elif pre[0] is None:
                outs[tag] = dict(zip(("f3", "mask_pred", "r1", "r2"), self._frozen_encoder_outputs(m, x)))
                outs[tag]["frozen"] = True
            else:
                outs[tag] = {"f3": pre[0], "mask_pred": pre[1], "frozen": True}
        enc_d = outs["dwi"] if trainable["dwi"] else None
        enc_c = outs["dce"] if trainable["dce"] else None
        f3d, f3c, md, mc = outs["dwi"]["f3"], outs["dce"]["f3"], outs["dwi"]["mask_pred"], outs["dce"]["mask_pred"]
        ops.tape.record(self._marker(6))
        fo = fusion_forward_train(ops, self.fusion, f3d, f3c, md, mc)
        total, parts = fusion_objective(ops, fo, enc_d, enc_c, masks, labels, dwi_in, dce_in, md=md, mc=mc, aux_w=self.aux_w,
                                        frozen_d=None if trainable["dwi"] else outs["dwi"],
                                        frozen_c=None if trainable["dce"] else outs["dce"], **self.loss_hp)
        self.flat["g"][self.flat_numel:].copy_(total)   # the loss rides along with the gradients
        ops.tape.backward()
        if self._reduced_from > 0:  # whatever is left
            self._reduce_range(0, self._reduced_from)
        if self._world() > 1:
            self._reduce_range(self.flat_numel, self.flat_numel + 1)
        self.logits = fo["logits"]
        self.fused_mask_logits = fo["fused_mask"]
        return total, parts

    def step(self):
        """Wait for the gradient exchange, then one fused AdamW launch over the flat buffer (per-element learning rate /
        weight decay / first step; grad_scale folds the 1 / world average).  Returns the rank-averaged loss."""
        world = self._world()
        if self._comm is not None:
            for w in self._pending:
                w.wait()
            torch.cuda.current_stream(self.dev).wait_stream(self._comm)
        self.step_count += 1
        f = self.flat
        _call("b200_adamw_groups", _P(f["p"]), _P(f["g"]), _P(f["m"]), _P(f["v"]), self.flat_numel, _P(f["lr"]), _P(f["wd"]),
              _P(f["step0"]), float(self.lr_mult), float(self.hp["betas"][0]), float(self.hp["betas"][1]),
              float(self.hp["eps"]), self.step_count, 1.0 / world, _s())
        return f["g"][self.flat_numel:] / world

    def train_step(self, dwi_in, dce_in, masks, labels, **kw):
        self.zero_grad()
        total, parts = self.forward_backward(dwi_in, dce_in, masks, labels, **kw)
        self.step()
        return total, parts


def _encoder_with_markers(ops, m, x, marks):
    """encoder_forward_train with all-reduce bucket markers at the forward positions of block1 / block2 / block3."""
    ops._bucket_marks = list(marks)
    try:
        return encoder_forward_train(ops, m, x, heads=False)
    finally:
        ops._bucket_marks = None


_NO_GRAD_PREFIXES_SINGLE = ("proj_r1.", "proj_r2.", "f2_to_f3.", "f2_weight", "f3_weight", "norm_f2.", "norm_f3.",
                            "mask_head.down_")


class SingleModelTrainer:
    """One optimisation step of LightningSingleModel (BASELINE config C1; code/train.py:294-428, AdamW
    code/selector_helpers.py:222-229) for one encoder: train-mode forward, the single-modality objective, explicit
    backward, one fused AdamW launch over a flat parameter buffer.  Parameters the objective cannot reach (the teacher
    projectors - the mimic term detaches them -, the unused aligner / backbone-mix parameters / mask-head
    down-samplers) stay outside the buffers, as torch.optim.AdamW skips parameters whose .grad is None."""

    def __init__(self, model, *, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=4e-5, smoothing=0.1, gamma=1.5,
                 class_weights=None, lambda_mask=0.2, lambda_recon=0.1, lambda_mimic=0.2, lambda_feat_norm=4e-5, seed=0x5EED):
        from fusion_train import flat_size, flat_views

        _check_supported(model)
        self.model = model
        self.hp = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.loss_hp = dict(smoothing=smoothing, gamma=gamma, class_weights=class_weights, lambda_mask=lambda_mask,
                            lambda_recon=lambda_recon, lambda_mimic=lambda_mimic, lambda_feat_norm=lambda_feat_norm)
        dev = next(model.parameters()).device
        if dev.type != "cuda":
            raise nat.B200NativeError("SingleModelTrainer needs the model on a CUDA device (no CPU path)")
        self.dev = dev
        self.ops = TrainOps(dev, drop_seed=seed)
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad and not n.startswith(_NO_GRAD_PREFIXES_SINGLE)]
        self.names = [n for n, _ in named]
        self.params = [p for _, p in named]
        self.numel = sum(p.numel() for p in self.params)
        n = flat_size(self.params)
        self.flat_numel = n
        self.flat = {k: torch.zeros(n, dtype=torch.float32, device=dev) for k in ("p", "g", "m", "v")}
        for p, view in zip(self.params, flat_views(self.params, self.flat["p"])):
            view.copy_(p.data.float())
            p.data = view
        for p, g in zip(self.params, flat_views(self.params, self.flat["g"])):
            p.grad = g
        self.step_count = 0

    def train_step(self, x, masks, labels):
        self.flat["g"].zero_()
        self.ops.new_step()
        out = encoder_forward_train(self.ops, self.model, x)
        total, parts = single_model_loss(self.ops, out, masks.to(self.dev).float(), labels.to(self.dev, torch.int64).contiguous(),
                                         **self.loss_hp)
        self.ops.tape.backward()
        self.step_count += 1
        f = self.flat
        nat.adamw(f["p"], f["g"], f["m"], f["v"], lr=self.hp["lr"], betas=self.hp["betas"], eps=self.hp["eps"],
                  weight_decay=self.hp["weight_decay"], step=self.step_count)
        self.logits = out["logits"]
        return total, parts


# ------------------------------------------------------------------------------------------------------------------
# torch.autograd bridge: lets code written against the reference modules - `loss = f(model(x)); loss.backward()`, i.e.
# the reference's own train.py / train_fusion.py `_shared_step` - drive the training kernels.  One autograd node per
# module forward; its backward seeds the tape with the incoming gradients and runs it.  Parameter gradients are
# accumulated by the kernels straight into `param.grad` (the node returns None for them).
# ------------------------------------------------------------------------------------------------------------------
def _to_map_grad(g, like):
    """Incoming autograd gradient -> the layout / dtype of the tape tensor `like` (NHWC bf16 map or fp32 vector)."""
    if g is None:
        return None
    return g.to(like.dtype).contiguous() if g.shape == like.shape else g.reshape(like.shape).to(like.dtype).contiguous()


class _EncoderTrainFn(torch.autograd.Function):
    KEYS = ("logits", "f1", "f2", "f3", "r1", "r2", "p1", "p1_r", "p2", "p2_r", "mask_pred")

    @staticmethod
    def forward(ctx, module, x, *params):
        ops = TrainOps(x.device, drop_seed=getattr(module, "_train_seed", 0x5EED))
        module._train_seed = (getattr(module, "_train_seed", 0x5EED) * 6364136223846793005 + 1442695040888963407) & 0xFFFFFFFFFFFF
        out = encoder_forward_train(ops, module, x)
        ctx.ops, ctx.out, ctx.n_params = ops, out, len(params)
        res = tuple(out[k] for k in _EncoderTrainFn.KEYS) + (out["mask_attn_map"], out["mod_attn_map"])
        ctx.mark_non_differentiable(res[-2], res[-1])
        return res

    @staticmethod
    def backward(ctx, *grads):
        tape = ctx.ops.tape
        for k, g in zip(_EncoderTrainFn.KEYS, grads):
            if g is not None:
                tape.add_grad(ctx.out[k], _to_map_grad(g, ctx.out[k]))
        tape.backward()
        return (None, None) + (None,) * ctx.n_params


class _FusionTrainFn(torch.autograd.Function):
    KEYS = ("logits", "fused_mask", "recon", "proj", "p_dwi", "p_dce")

    @staticmethod
    def forward(ctx, module, f3d, f3c, md, mc, *params):
        ops = TrainOps(f3d.device)
        fo = fusion_forward_train(ops, module, f3d, f3c, md, mc)
        ctx.ops, ctx.fo, ctx.inputs, ctx.n_params = ops, fo, (f3d, f3c, md, mc), len(params)
        res = tuple(fo[k] for k in _FusionTrainFn.KEYS) + (fo["gating"],)
        ctx.mark_non_differentiable(res[-1])
        return res

    @staticmethod
    def backward(ctx, *grads):
        tape = ctx.ops.tape
        for k, g in zip(_FusionTrainFn.KEYS, grads):
            if g is not None:
                tape.add_grad(ctx.fo[k], _to_map_grad(g, ctx.fo[k]))
        want = [t for t in ctx.inputs if t is not None]
        got = iter(tape.backward(want))
        gin = tuple(next(got) if t is not None else None for t in ctx.inputs)
        return (None,) + gin + (None,) * ctx.n_params


def encoder_train_forward_autograd(module, x):
    """ModelMaskHeadBackbone.forward in training mode with torch-autograd semantics: returns the reference's
    (logits, aux, mask_pred) whose tensors carry a grad_fn."""
    params = [p for p in module.parameters() if p.requires_grad]
    x = x.contiguous().float()
    if not params:  # nothing to differentiate: still the train-mode arithmetic (batch statistics, dropout)
        ops = TrainOps(x.device)
        out = encoder_forward_train(ops, module, x)
        ops.tape.steps.clear()
        res = tuple(out[k] for k in _EncoderTrainFn.KEYS) + (out["mask_attn_map"], out["mod_attn_map"])
    else:
        res = _EncoderTrainFn.apply(module, x, *params)
    logits, f1, f2, f3, r1, r2, p1, p1_r, p2, p2_r, mask_pred, attn, mod = res
    nchw = lambda t: t.permute(0, 3, 1, 2)
    pd = module.proj_dim

    def pooled(t):  # AdaptiveAvgPool2d((proj_dim, proj_dim)) of the reference ahead of the projector: a 2x2 replication
        t = nchw(t)
        if t.shape[-1] == pd:
            return t
        if pd == 2 * t.shape[-1]:
            return t.repeat_interleave(2, dim=2).repeat_interleave(2, dim=3)
        raise NotImplementedError("training path: proj_dim equal to or twice the map size")

    B, C = x.shape[:2]
    aux = {"raw_feats": [nchw(f1), nchw(f2), nchw(f3)], "recon_feats": [r1.unsqueeze(1), r2.unsqueeze(1)],
           "proj_pairs": [pooled(p1), pooled(p1_r), pooled(p2), pooled(p2_r)], "mask_attn_map": attn.unsqueeze(1),
           "mod_attn_map": mod.view(B, C, 1, 1)}
    return logits, aux, mask_pred.unsqueeze(1)


def fusion_train_forward_autograd(module, raw_feats_dwi, raw_feats_dce, dwi_mask_pred, dce_mask_pred):
    """FusionModel.forward in training mode with torch-autograd semantics."""
    def nhwc(t):
        v = t.permute(0, 2, 3, 1)
        return v if (v.dtype == torch.bfloat16 and v.is_contiguous()) else v.to(torch.bfloat16).contiguous()

    f3d, f3c = nhwc(raw_feats_dwi[-1]), nhwc(raw_feats_dce[-1])
    md = dwi_mask_pred[:, 0].contiguous().float() if dwi_mask_pred is not None else None
    mc = dce_mask_pred[:, 0].contiguous().float() if dce_mask_pred is not None else None
    params = [p for p in module.parameters() if p.requires_grad]
    res = _FusionTrainFn.apply(module, f3d, f3c, md, mc, *params)
    logits, fused_mask, recon, proj, p_dwi, p_dce, gating = res
    nchw = lambda t: t.permute(0, 3, 1, 2)
    aux = {"proj_fused": nchw(proj), "recon_fused": recon.unsqueeze(1), "gating_weights": gating, "attn_weights": None,
           "p_dwi": nchw(p_dwi), "p_dce": nchw(p_dce)}
    return logits, fused_mask.unsqueeze(1), aux
