"""Reference-compatible parameter layout of the U-Net.

The drop-in boundary includes the ``state_dict`` contract (SURVEY.md section 8b): a
checkpoint written by the reference's ``Unet`` must load unchanged.  Instead of
re-declaring the reference's module classes, the layout is *generated* from the
constructor kwargs as a flat ``key -> (shape, init)`` table and then hung on a tree of
anonymous ``nn.Module`` containers so that ``state_dict()`` / ``load_state_dict()``
produce and accept exactly the reference's dotted keys
(reference constructor: imagen_pytorch.py:1113-1442; tests/test_params.py checks the
table against the key/shape contract dumped from the live reference).
"""
from __future__ import annotations

import math
from collections import OrderedDict

import torch
from torch import nn


def cast_tuple(val, length=1):
    if isinstance(val, list):
        val = tuple(val)
    out = val if isinstance(val, tuple) else (val,) * length
    return out


UNET_DEFAULTS = OrderedDict(
    dim=None, text_embed_dim=768, num_resnet_blocks=1, cond_dim=None, num_image_tokens=4,
    num_time_tokens=2, learned_sinu_pos_emb_dim=16, out_dim=None, dim_mults=(1, 2, 4, 8),
    cond_images_channels=0, channels=3, channels_out=None, attn_dim_head=64, attn_heads=8,
    ff_mult=2., lowres_cond=False, layer_attns=True, layer_attns_depth=1, layer_mid_attns_depth=1,
    layer_attns_add_text_cond=True, attend_at_middle=True, layer_cross_attns=True,
    use_linear_attn=False, use_linear_cross_attn=False, cond_on_text=True, max_text_len=256,
    init_dim=None, init_conv_kernel_size=7, init_cross_embed=True,
    init_cross_embed_kernel_sizes=(3, 7, 15), cross_embed_downsample=False,
    cross_embed_downsample_kernel_sizes=(2, 4), attn_pool_text=True, attn_pool_num_latents=32,
    dropout=0., memory_efficient=False, init_conv_to_final_conv_residual=False,
    use_global_context_attn=True, scale_skip_connection=True, final_resnet_block=True,
    final_conv_kernel_size=3, self_cond=False, resize_mode='nearest',
    combine_upsample_fmaps=False, pixel_shuffle_upsample=True,
)

# Options of the reference constructor that this hot-path implementation does not cover.
# They raise instead of silently diverging (SURVEY.md section 7 "API edge cases").
_UNSUPPORTED = dict(
    use_linear_attn=lambda v: any(cast_tuple(v)),
    cross_embed_downsample=bool,
    combine_upsample_fmaps=bool, init_conv_to_final_conv_residual=bool,
    pixel_shuffle_upsample=lambda v: not v, attn_dim_head=lambda v: v > 64 or v < 1,
    final_resnet_block=lambda v: not v,
)


class UnetArch:
    """Resolved architecture: every derived dimension of Unet.__init__ (imagen_pytorch.py:1177-1436)."""

    def __init__(self, **kwargs):
        cfg = OrderedDict(UNET_DEFAULTS)
        for k, v in kwargs.items():
            if k not in cfg:
                raise TypeError(f"Unet() got an unexpected keyword argument '{k}'")
            cfg[k] = v
        if cfg['dim'] is None:
            raise TypeError("Unet() missing required keyword argument 'dim'")
        for k, bad in _UNSUPPORTED.items():
            if bad(cfg[k]):
                raise NotImplementedError(
                    f'imagen_pytorch_b200.Unet: {k}={cfg[k]!r} is outside the B200 sampling hot path '
                    f'(see DESIGN.md "out of scope"); use the reference implementation for it.')
        assert cfg['attn_heads'] > 1, 'you need to have more than 1 attention head, ideally at least 4 or 8'
        self.cfg = cfg
        g = cfg.__getitem__
        self.dim = g('dim')
        self.channels = g('channels')
        self.channels_out = g('channels_out') if g('channels_out') is not None else g('channels')
        self.lowres_cond = bool(g('lowres_cond'))
        self.cond_on_text = bool(g('cond_on_text'))
        self.self_cond = bool(g('self_cond'))
        self.cond_images_channels = int(g('cond_images_channels'))
        self.init_channels = self.channels * (1 + int(self.lowres_cond) + int(self.self_cond)) + self.cond_images_channels   # :1184, :1194
        self.init_dim = g('init_dim') if g('init_dim') is not None else self.dim
        self.dims = [self.init_dim, *[self.dim * m for m in g('dim_mults')]]
        self.in_out = list(zip(self.dims[:-1], self.dims[1:]))
        self.num_levels = len(self.in_out)
        self.cond_dim = g('cond_dim') if g('cond_dim') is not None else self.dim
        self.time_cond_dim = self.dim * 4 * (2 if self.lowres_cond else 1)
        self.num_time_tokens = g('num_time_tokens')
        self.sinu_dim = g('learned_sinu_pos_emb_dim')
        self.heads = g('attn_heads')
        self.dim_head = g('attn_dim_head')
        self.inner = self.heads * self.dim_head
        self.ff_mult = g('ff_mult')
        self.max_text_len = g('max_text_len')
        self.text_embed_dim = g('text_embed_dim')
        self.attn_pool = bool(g('attn_pool_text'))
        self.pool_latents = g('attn_pool_num_latents')
        self.pool_mean_latents = 4
        self.pool_depth = 2
        self.memory_efficient = bool(g('memory_efficient'))
        self.use_gca = bool(g('use_global_context_attn'))
        self.skip_scale = 2 ** -0.5 if g('scale_skip_connection') else 1.
        n = self.num_levels
        self.num_resnet_blocks = cast_tuple(g('num_resnet_blocks'), n)
        self.layer_attns = cast_tuple(g('layer_attns'), n)
        self.layer_attns_depth = cast_tuple(g('layer_attns_depth'), n)
        self.layer_cross_attns = cast_tuple(g('layer_cross_attns'), n)
        self.use_linear_cross_attn = cast_tuple(g('use_linear_cross_attn'), n)
        assert len(self.layer_attns) == n and len(self.layer_cross_attns) == n and len(self.num_resnet_blocks) == n
        assert len(self.use_linear_cross_attn) == n
        self.mid_depth = g('layer_mid_attns_depth')
        self.attend_at_middle = bool(g('attend_at_middle'))
        self.init_cross_embed = bool(g('init_cross_embed'))
        self.init_kernels = tuple(sorted(g('init_cross_embed_kernel_sizes'))) if self.init_cross_embed else (g('init_conv_kernel_size'),)
        if self.init_cross_embed:
            ns = len(self.init_kernels)
            ds = [int(self.init_dim / (2 ** i)) for i in range(1, ns)]
            self.init_dim_scales = [*ds, self.init_dim - sum(ds)]
        else:
            self.init_dim_scales = [self.init_dim]
        self.final_kernel = g('final_conv_kernel_size')
        if self.dim % 8 != 0 or self.init_dim % 8 != 0 or self.cond_dim % 8 != 0:
            raise NotImplementedError('imagen_pytorch_b200.Unet needs dim / init_dim / cond_dim to be multiples of 8 (16-byte NHWC rows)')

    # level-wise channel bookkeeping ------------------------------------------------------------
    def _cross(self, i):
        """A level has a cross-attention layer when either flag asks for one; use_linear_cross_attn picks LinearCrossAttention
        (imagen_pytorch.py:1341, :1370, :1395, :1409), which has CrossAttention's parameters."""
        lin = bool(self.use_linear_cross_attn[i])
        return dict(cross=bool(self.layer_cross_attns[i]) or lin, linear_cross=lin)

    def down_level(self, i):
        dim_in, dim_out = self.in_out[i]
        cur = dim_out if self.memory_efficient else dim_in
        return dict(dim_in=dim_in, dim_out=dim_out, cur=cur, is_last=i >= self.num_levels - 1, **self._cross(i), attn=bool(self.layer_attns[i]),
                    depth=self.layer_attns_depth[i], nres=self.num_resnet_blocks[i])

    def up_level(self, i):
        lev = self.num_levels - 1 - i
        dim_in, dim_out = self.in_out[lev]
        skip = self.down_level(lev)['cur']
        return dict(lev=lev, dim_in=dim_in, dim_out=dim_out, skip=skip, is_last=i == self.num_levels - 1, **self._cross(lev), attn=bool(self.layer_attns[lev]),
                    depth=self.layer_attns_depth[lev], nres=self.num_resnet_blocks[lev])


# ----------------------------------------------------------------------------------------------
# key -> (shape, init) table.  init kinds: 'w' (kaiming-uniform-like), 'b' (uniform bias, fan_in
# in the tuple), 'ones', 'zeros', 'randn', 'ps' (pixel-shuffle ICNR-style repeat, :621-628)
# ----------------------------------------------------------------------------------------------

def param_table(a: UnetArch):
    t = OrderedDict()

    def conv(p, cout, cin, k):
        t[p + '.weight'] = ((cout, cin, k, k), 'w')
        t[p + '.bias'] = ((cout,), ('b', cin * k * k))

    def linear(p, cout, cin, bias=True):
        t[p + '.weight'] = ((cout, cin), 'w')
        if bias:
            t[p + '.bias'] = ((cout,), ('b', cin))

    def nn_ln(p, d):
        t[p + '.weight'] = ((d,), 'ones')
        t[p + '.bias'] = ((d,), 'zeros')

    def feedforward(p, d, mult):                                   # :972-980
        hid = int(d * mult)
        t[p + '.0.g'] = ((d,), 'ones')
        linear(p + '.1', hid, d, bias=False)
        t[p + '.3.g'] = ((hid,), 'ones')
        linear(p + '.4', d, hid, bias=False)

    def resnet(p, din, dout, cond_dim=None, use_gca=False, heads=a.heads, dim_head=a.dim_head):   # :693-733
        linear(p + '.time_mlp.1', dout * 2, a.time_cond_dim)
        if cond_dim is not None:
            inner = heads * dim_head
            c = p + '.cross_attn'
            t[c + '.null_kv'] = ((2, dim_head), 'randn')
            t[c + '.q_scale'] = ((dim_head,), 'ones')
            t[c + '.k_scale'] = ((dim_head,), 'ones')
            t[c + '.norm.g'] = ((dout,), 'ones')
            linear(c + '.to_q', inner, dout, bias=False)
            linear(c + '.to_kv', inner * 2, cond_dim, bias=False)
            linear(c + '.to_out.0', dout, inner, bias=False)
            t[c + '.to_out.1.g'] = ((dout,), 'ones')
        t[p + '.block1.norm.gamma'] = ((din, 1, 1), 'ones')
        conv(p + '.block1.project', dout, din, 3)
        t[p + '.block2.norm.gamma'] = ((dout, 1, 1), 'ones')
        conv(p + '.block2.project', dout, dout, 3)
        if use_gca:
            hid = max(3, dout // 2)
            conv(p + '.gca.to_k', 1, dout, 1)
            conv(p + '.gca.net.0', hid, dout, 1)
            conv(p + '.gca.net.2', dout, hid, 1)
        if din != dout:
            conv(p + '.res_conv', dout, din, 1)

    def transformer(p, d, depth, context_dim):                     # :992-1010, :502-532
        for l in range(depth):
            q = f'{p}.layers.{l}.0'
            t[q + '.null_kv'] = ((2, a.dim_head), 'randn')
            t[q + '.q_scale'] = ((a.dim_head,), 'ones')
            t[q + '.k_scale'] = ((a.dim_head,), 'ones')
            t[q + '.norm.g'] = ((d,), 'ones')
            linear(q + '.to_q', a.inner, d, bias=False)
            linear(q + '.to_kv', a.dim_head * 2, d, bias=False)
            if context_dim is not None:
                nn_ln(q + '.to_context.0', context_dim)
                linear(q + '.to_context.1', a.dim_head * 2, context_dim)
            linear(q + '.to_out.0', d, a.inner, bias=False)
            t[q + '.to_out.1.g'] = ((d,), 'ones')
            feedforward(f'{p}.layers.{l}.1', d, a.ff_mult)

    # ---- stem / conditioning (:1198-1287)
    if a.init_cross_embed:
        for i, (k, ds) in enumerate(zip(a.init_kernels, a.init_dim_scales)):
            conv(f'init_conv.convs.{i}', ds, a.init_channels, k)
    else:
        conv('init_conv', a.init_dim, a.init_channels, a.init_kernels[0])
    t['to_time_hiddens.0.weights'] = ((a.sinu_dim // 2,), 'randn')
    linear('to_time_hiddens.1', a.time_cond_dim, a.sinu_dim + 1)
    linear('to_time_cond.0', a.time_cond_dim, a.time_cond_dim)
    linear('to_time_tokens.0', a.cond_dim * a.num_time_tokens, a.time_cond_dim)
    if a.lowres_cond:
        t['to_lowres_time_hiddens.0.weights'] = ((a.sinu_dim // 2,), 'randn')
        linear('to_lowres_time_hiddens.1', a.time_cond_dim, a.sinu_dim + 1)
        linear('to_lowres_time_cond.0', a.time_cond_dim, a.time_cond_dim)
        linear('to_lowres_time_tokens.0', a.cond_dim * a.num_time_tokens, a.time_cond_dim)
    nn_ln('norm_cond', a.cond_dim)
    if a.cond_on_text:
        assert a.text_embed_dim is not None, 'text_embed_dim must be given to the unet if cond_on_text is True'
        linear('text_to_cond', a.cond_dim, a.text_embed_dim)
    if a.attn_pool:                                                # PerceiverResampler :447-479
        p = 'attn_pool'
        t[p + '.pos_emb.weight'] = ((512, a.cond_dim), 'randn')
        t[p + '.latents'] = ((a.pool_latents, a.cond_dim), 'randn')
        t[p + '.to_latents_from_mean_pooled_seq.0.g'] = ((a.cond_dim,), 'ones')
        linear(p + '.to_latents_from_mean_pooled_seq.1', a.cond_dim * a.pool_mean_latents, a.cond_dim)
        for l in range(a.pool_depth):
            q = f'{p}.layers.{l}.0'
            nn_ln(q + '.norm', a.cond_dim)
            nn_ln(q + '.norm_latents', a.cond_dim)
            linear(q + '.to_q', a.inner, a.cond_dim, bias=False)
            linear(q + '.to_kv', a.inner * 2, a.cond_dim, bias=False)
            t[q + '.q_scale'] = ((a.dim_head,), 'ones')
            t[q + '.k_scale'] = ((a.dim_head,), 'ones')
            linear(q + '.to_out.0', a.cond_dim, a.inner, bias=False)
            nn_ln(q + '.to_out.1', a.cond_dim)
            feedforward(f'{p}.layers.{l}.1', a.cond_dim, 4)
    t['null_text_embed'] = ((1, a.max_text_len, a.cond_dim), 'randn')
    t['null_text_hidden'] = ((1, a.time_cond_dim), 'randn')
    if a.cond_on_text:
        nn_ln('to_text_non_attn_cond.0', a.cond_dim)
        linear('to_text_non_attn_cond.1', a.time_cond_dim, a.cond_dim)
        linear('to_text_non_attn_cond.3', a.time_cond_dim, a.time_cond_dim)

    # ---- body (:1319-1413)
    if a.memory_efficient:
        resnet('init_resnet_block', a.init_dim, a.init_dim, use_gca=a.use_gca)
    for i in range(a.num_levels):
        L = a.down_level(i)
        p = f'downs.{i}'
        if a.memory_efficient:
            conv(p + '.0.1', L['dim_out'], L['dim_in'] * 4, 1)
        resnet(p + '.1', L['cur'], L['cur'], cond_dim=a.cond_dim if L['cross'] else None)
        for j in range(L['nres']):
            resnet(f'{p}.2.{j}', L['cur'], L['cur'], use_gca=a.use_gca)
        if L['attn']:
            transformer(p + '.3', L['cur'], L['depth'], a.cond_dim)
        if not a.memory_efficient:
            if not L['is_last']:
                conv(p + '.4.1', L['dim_out'], L['cur'] * 4, 1)
            else:
                conv(p + '.4.fns.0', L['dim_out'], L['dim_in'], 3)
                conv(p + '.4.fns.1', L['dim_out'], L['dim_in'], 1)
    mid = a.dims[-1]
    resnet('mid_block1', mid, mid, cond_dim=a.cond_dim, heads=8, dim_head=64)     # plain ResnetBlock: default heads/dim_head (:1380)
    if a.attend_at_middle:
        transformer('mid_attn', mid, a.mid_depth, None)
    resnet('mid_block2', mid, mid, cond_dim=a.cond_dim, heads=8, dim_head=64)
    for i in range(a.num_levels):
        U = a.up_level(i)
        p = f'ups.{i}'
        resnet(p + '.0', U['dim_out'] + U['skip'], U['dim_out'], cond_dim=a.cond_dim if U['cross'] else None)
        for j in range(U['nres']):
            resnet(f'{p}.1.{j}', U['dim_out'] + U['skip'], U['dim_out'], use_gca=a.use_gca)
        if U['attn']:
            transformer(p + '.2', U['dim_out'], U['depth'], a.cond_dim)
        if (not U['is_last']) or a.memory_efficient:
            t[p + '.3.net.0.weight'] = ((U['dim_in'] * 4, U['dim_out'], 1, 1), 'ps')
            t[p + '.3.net.0.bias'] = ((U['dim_in'] * 4,), 'zeros')
    resnet('final_res_block', a.dim, a.dim, use_gca=True)
    fin = a.dim + (a.channels if a.lowres_cond else 0)
    t['final_conv.weight'] = ((a.channels_out, fin, a.final_kernel, a.final_kernel), 'zeros')   # zero_init_ :1438
    t['final_conv.bias'] = ((a.channels_out,), 'zeros')
    return t


def _init_tensor(shape, kind):
    if kind == 'ones':
        return torch.ones(shape)
    if kind == 'zeros':
        return torch.zeros(shape)
    if kind == 'randn':
        return torch.randn(shape)
    if kind == 'w':
        fan_in = 1
        for d in shape[1:]:
            fan_in *= d
        bound = 1 / math.sqrt(fan_in)
        return torch.empty(shape).uniform_(-bound, bound)
    if kind == 'ps':
        o, i, h, w = shape
        bound = math.sqrt(6 / (i * h * w)) / math.sqrt(1 + 5)   # kaiming_uniform_(a=0) bound scaled like nn.init default gain
        base = torch.empty(o // 4, i, h, w).uniform_(-bound * math.sqrt(3), bound * math.sqrt(3))
        return base.repeat_interleave(4, dim=0)                    # 'o ... -> (o 4) ...'
    if isinstance(kind, tuple) and kind[0] == 'b':
        bound = 1 / math.sqrt(kind[1])
        return torch.empty(shape).uniform_(-bound, bound)
    raise ValueError(kind)


class ParamNode(nn.Module):
    """Anonymous container: exists only so dotted state_dict keys match the reference."""


def build_param_tree(root: nn.Module, table):
    for key, (shape, kind) in table.items():
        parts = key.split('.')
        node = root
        for name in parts[:-1]:
            child = node._modules.get(name)
            if child is None:
                child = ParamNode()
                node.add_module(name, child)
            node = child
        node.register_parameter(parts[-1], nn.Parameter(_init_tensor(shape, kind)))


# ----------------------------------------------------------------------------------------------
# attention head width.  The sm_100a attention kernels work on 64-wide heads (one 128-byte swizzle row per key).  Narrower heads
# (the reference's UnetConfig defaults to attn_dim_head=32, configs.py:49-50) run on the same kernels with every head zero-padded
# to 64 channels: q.k, the L2 norms and P.V are unchanged by zero channels, and the padded output channels meet zero columns of
# to_out.  Only the packed operands are padded -- the module's state_dict keeps the reference layout.
# ----------------------------------------------------------------------------------------------
HEAD_PAD = 64
_PAD_DIM0 = ('.to_q.weight', '.to_kv.weight', '.to_context.1.weight', '.to_context.1.bias', '.q_scale', '.k_scale')


def pad_attention_heads(sd, dim_head):
    """{key: tensor} of every attention parameter of `sd` (host tensors) re-laid out for 64-wide heads; {} when dim_head == 64."""
    if dim_head == HEAD_PAD:
        return {}
    assert dim_head < HEAD_PAD
    out = {}
    for k, v in sd.items():
        if k.startswith(('mid_block1.', 'mid_block2.')):      # plain ResnetBlock(mid_dim): CrossAttention defaults heads=8, dim_head=64 (:1380, :1382)
            continue
        if k.endswith(_PAD_DIM0) and ('attn' in k or '.layers.' in k):
            assert v.shape[0] % dim_head == 0, (k, tuple(v.shape))
            g = v.reshape(v.shape[0] // dim_head, dim_head, *v.shape[1:])
            p = g.new_zeros(g.shape[0], HEAD_PAD, *g.shape[2:])
            p[:, :dim_head] = g
            out[k] = p.reshape(g.shape[0] * HEAD_PAD, *g.shape[2:]).contiguous()
        elif k.endswith('.null_kv'):
            p = v.new_zeros(*v.shape[:-1], HEAD_PAD)
            p[..., :dim_head] = v
            out[k] = p.contiguous()
        elif k.endswith('.to_out.0.weight') and v.ndim == 2 and v.shape[1] % dim_head == 0 and ('attn' in k or '.layers.' in k):
            g = v.reshape(v.shape[0], v.shape[1] // dim_head, dim_head)
            p = g.new_zeros(g.shape[0], g.shape[1], HEAD_PAD)
            p[..., :dim_head] = g
            out[k] = p.reshape(g.shape[0], -1).contiguous()
    return out
