"""Pins the linear cross-attention oracle (oracle/linear_cross_ref.py) against the LIVE reference and writes
tests/golden/linear_cross_attn_dim32.pt -- the only file it writes.

Run in the build container only, like oracle/make_golden.py (it uses the same import shim for the reference):
    python -m oracle.make_golden_linear_cross
Hard asserts at generation time: oracle == reference Unet.forward (cond / null / CFG-3) to 1e-5 * max|ref| for three architectures,
and oracle == reference Imagen.sample for a 6-step CFG DDPM trajectory.
"""
from __future__ import annotations

import os

import torch

from oracle import unet_ref, sampler_ref, linear_cross_ref
from oracle.make_golden import _install_shim, _maxdiff


LINEAR_CROSS_CASES = {
    # a linear-only level, a regular level, a linear level that also has layer_cross_attns=True; the mid blocks stay CrossAttention
    'A': dict(dim=32, dim_mults=(1, 2, 4), text_embed_dim=64, max_text_len=24, layer_attns=(False, False, True),
              layer_cross_attns=(False, True, True), use_linear_cross_attn=(True, False, True)),
    # zero-padded 32-wide heads, lowres time tokens in the context
    'B': dict(dim=32, dim_mults=(1, 2, 4), text_embed_dim=64, max_text_len=24, attn_dim_head=32, attn_heads=4, use_linear_cross_attn=True,
              lowres_cond=True, memory_efficient=True),
    # no text: the context is the two time tokens (three keys with the null)
    'C': dict(dim=32, dim_mults=(1, 2, 4), text_embed_dim=64, use_linear_cross_attn=True, cond_on_text=False),
}


def main():
    """Unet(use_linear_cross_attn=...) (LinearCrossAttention, imagen_pytorch.py:836-874): forward passes of three architectures and a
    6-step CFG DDPM trajectory -> tests/golden/linear_cross_attn_dim32.pt.  Weights and inputs are rebuilt from the stored seeds."""
    _install_shim()
    import imagen_pytorch as ref
    torch.set_num_threads(8)
    out = dict(cases=LINEAR_CROSS_CASES, contracts={}, outs={})
    B = 2
    g = torch.Generator().manual_seed(211)
    x = torch.randn(B, 3, 32, 32, generator=g)
    t = torch.tensor([-0.9, 1.1])
    te = torch.randn(B, 24, 64, generator=g)
    te[0, 11:] = 0.                                   # ragged text -> mask has False entries
    tm = torch.any(te != 0., dim=-1)
    low = torch.randn(B, 3, 32, 32, generator=g)
    lnt = torch.tensor([0.31, 0.62])
    out.update(x=x, t=t, text_embeds=te, text_mask=tm, lowres_cond_img=low, lowres_noise_times=lnt)
    for i, (name, kw) in enumerate(LINEAR_CROSS_CASES.items()):
        torch.manual_seed(0)
        u = ref.Unet(**kw)
        shapes = {k: tuple(v.shape) for k, v in u.state_dict().items()}
        sd = unet_ref.synth_state_dict(shapes, seed=300 + i)
        u.load_state_dict(sd)
        u.eval()
        cfg = unet_ref.unet_config(**kw)
        args = dict(text_embeds=te, text_mask=tm) if kw.get('cond_on_text', True) else {}
        if kw.get('lowres_cond'):
            args.update(lowres_cond_img=low, lowres_noise_times=lnt)
        with torch.no_grad(), linear_cross_ref.linear_layers(cfg):
            r = dict(cond=u(x, t, **args))
            o = dict(cond=unet_ref.unet_forward(sd, cfg, x, t, **args))
            if kw.get('cond_on_text', True):
                r['null'] = u(x, t, cond_drop_prob=1., **args)
                r['cfg3'] = u.forward_with_cond_scale(x, t, cond_scale=3., **args)
                o['null'] = unet_ref.unet_forward(sd, cfg, x, t, cond_drop_prob=1., **args)
                o['cfg3'] = unet_ref.unet_forward_with_cond_scale(sd, cfg, x, t, cond_scale=3., **args)
        for k in r:
            d = _maxdiff(r[k], o[k])
            print(f'[linear cross {name} {k}] ref-vs-oracle max|d| = {d:.3e}  (|ref|max {r[k].abs().max():.3f})')
            assert d < 1e-5 * max(1., r[k].abs().max().item()), (name, k)
        out['contracts'][name] = shapes
        out['outs'][name] = dict(wseed=300 + i, **r)
        if name == 'A':
            im = ref.Imagen(unets=u, image_sizes=32, timesteps=6, text_embed_dim=64)
            im.unets[0].load_state_dict(sd)
            torch.manual_seed(223)
            r_img = im.sample(text_embeds=te, cond_scale=3., use_tqdm=False)
            torch.manual_seed(223)
            with linear_cross_ref.linear_layers(cfg):
                o_img = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=te, timesteps=6, cond_scale=3.)
            d = _maxdiff(r_img, o_img)
            print(f'[linear cross A ddpm sample] ref-vs-oracle max|d| = {d:.3e}')
            assert d < 1e-4
            out['sample'] = dict(seed=223, timesteps=6, cond_scale=3., out=r_img)
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden', 'linear_cross_attn_dim32.pt')
    torch.save(out, path)
    print(path, os.path.getsize(path) // 1024, 'KiB')


if __name__ == '__main__':
    main()
