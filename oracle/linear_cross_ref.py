"""ORACLE (test infrastructure, NOT product code) -- LinearCrossAttention (imagen_pytorch.py:836-874) for
Unet(use_linear_cross_attn=...), in CPU / GPU torch fp32.

The flag only changes which attention a level's ResnetBlock builds (:719, :1370, :1409); the parameters are CrossAttention's,
so oracle.unet_ref.unet_forward runs these models unchanged once its cross-attention dispatches on the layer.  `linear_layers`
does that for the duration of a `with` block: every oracle.unet_ref / oracle.sampler_ref call inside it runs the linear
layers of `cfg` through `linear_cross_attention`.  Pinned against the live reference by oracle/make_golden_linear_cross.py.
"""
from __future__ import annotations

import contextlib

import torch
import torch.nn.functional as F

from . import unet_ref


def linear_cross_attention(x, context, sd, p, heads):   # LinearCrossAttention.forward (the mask branch is unused: :749 passes none)
    b = x.shape[0]
    x = unet_ref._ln_gain(x, sd[p + '.norm.g'])
    q = F.linear(x, sd[p + '.to_q.weight'])
    k, v = F.linear(context, sd[p + '.to_kv.weight']).chunk(2, dim=-1)
    q, k, v = (unet_ref._split_heads(t, heads) for t in (q, k, v))
    nk, nv = sd[p + '.null_kv'].unbind(dim=-2)
    k = torch.cat((nk.expand(b, heads, 1, -1), k), dim=-2)
    v = torch.cat((nv.expand(b, heads, 1, -1), v), dim=-2)
    q = q.softmax(dim=-1) * 8                         # CrossAttention's scale = 8; no l2norm, q_scale / k_scale unused
    k = k.softmax(dim=-2)
    ctx = torch.einsum('bhnd,bhne->bhde', k, v)
    out = unet_ref._merge_heads(torch.einsum('bhnd,bhde->bhne', q, ctx))
    out = F.linear(out, sd[p + '.to_out.0.weight'])
    return unet_ref._ln_gain(out, sd[p + '.to_out.1.g'])


def linear_prefixes(cfg):
    """'<block>.cross_attn' of every LinearCrossAttention layer: the first ResnetBlock of each flagged down level and of its up level."""
    nlev = len(cfg['dim_mults'])
    lin = unet_ref._tup(cfg.get('use_linear_cross_attn', False), nlev)
    out = {f'downs.{i}.1.cross_attn' for i in range(nlev) if lin[i]}
    out |= {f'ups.{nlev - 1 - i}.0.cross_attn' for i in range(nlev) if lin[i]}
    return out


@contextlib.contextmanager
def linear_layers(cfg):
    linear = linear_prefixes(cfg)
    regular = unet_ref._cross_attention

    def dispatch(x, context, sd, p, heads):
        return (linear_cross_attention if p in linear else regular)(x, context, sd, p, heads)

    unet_ref._cross_attention = dispatch
    try:
        yield
    finally:
        unet_ref._cross_attention = regular
