"""fp32 CPU oracle of the hybrid TransformerStage in MC-dropout inference (test infrastructure only).

oracle/model_oracle.py restates the stage in eval mode, where every Dropout is identity.  This module restates it with
the blocks' nn.Dropout layers active (torch's global generator), and runs oracle/model_oracle.encoder_forward with that
stage in place.  The reference's TransformerStage source is not in this tree, so the placement follows its module
structure - MultiHeadSelfAttention(attn_drop=0.1, proj_drop=0.1) and MLP(drop=0.1) with a single `drop` module,
transformer_model.py:98-116, :128-134 - under timm's convention, which those names follow, and SURVEY.md a14
("dropout 0.1 everywhere"):
  1. attn_drop on the softmax probabilities, before `@ v` (row sums of the undropped softmax);
  2. proj_drop on proj(o), before LayerScale and the residual;
  3. MLP.drop after the GELU;
  4. MLP.drop again after fc2, before LayerScale and the residual.
With drop_p = 0 this is oracle/model_oracle.transformer_stage bit for bit (tests/test_mc_dropout_hybrid_cpu.py).
"""
from __future__ import annotations

import torch.nn.functional as F

from oracle import model_oracle as mo

TRANSFORMER_DROPOUT = 0.1  # the constructor defaults, as in the package's drop-in transformer_model.py (:109, :130)


def _drop(t, p):
    return F.dropout(t, p, training=p > 0)


def mhsa(x, s, heads, drop_p):
    """transformer_model.py:98-116 with attn_drop / proj_drop (places 1, 2)."""
    b, n, c = x.shape
    dh = c // heads
    qkv = F.linear(x, s["qkv.weight"], s["qkv.bias"]).reshape(b, n, 3, heads, dh).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    attn = _drop(((q @ k.transpose(-2, -1)) * dh ** -0.5).softmax(dim=-1), drop_p)
    y = (attn @ v).transpose(1, 2).reshape(b, n, c)
    return _drop(F.linear(y, s["proj.weight"], s["proj.bias"]), drop_p)


def transformer_stage(x, s, heads, patch, drop_p=0.0):
    """transformer_model.py:137-175 with every block's Dropouts at drop_p (places 1-4)."""
    pe = s.sub("patch_embed")
    t = F.conv2d(x, pe["proj.weight"], pe["proj.bias"], stride=patch)
    hs, ws = t.shape[-2:]
    t = t.flatten(2).transpose(1, 2)
    e = t.shape[-1]
    t = F.layer_norm(t, (e,), pe["norm.weight"], pe["norm.bias"])
    i = 0
    while s.has(f"transformer.layers.{i}.norm1.weight"):
        l = s.sub(f"transformer.layers.{i}")
        h = F.layer_norm(t, (e,), l["norm1.weight"], l["norm1.bias"])
        t = t + mhsa(h, l.sub("attn"), heads, drop_p) * l["gamma1"]
        h = F.layer_norm(t, (e,), l["norm2.weight"], l["norm2.bias"])
        h = _drop(F.gelu(F.linear(h, l["mlp.fc1.weight"], l["mlp.fc1.bias"])), drop_p)
        h = _drop(F.linear(h, l["mlp.fc2.weight"], l["mlp.fc2.bias"]), drop_p)
        t = t + h * l["gamma2"]
        i += 1
    return t.transpose(1, 2).reshape(x.shape[0], e, hs, ws)


def encoder_forward(sd, method, params, x, mc_dropout=False, transformer_dropout=None):
    """oracle/model_oracle.encoder_forward with the CNN blocks' Dropouts active when mc_dropout (p = the config's
    dropout) and the hybrid stage's active when transformer_dropout (p = 0.1; None follows mc_dropout)."""
    on = mc_dropout if transformer_dropout is None else transformer_dropout
    p = TRANSFORMER_DROPOUT if on else 0.0
    eval_stage = mo.transformer_stage
    mo.transformer_stage = lambda x_, s_, heads, patch: transformer_stage(x_, s_, heads, patch, p)
    try:
        return mo.encoder_forward(sd, method, params, x, mc_dropout=mc_dropout)
    finally:
        mo.transformer_stage = eval_stage
