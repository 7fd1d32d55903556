"""Pins the oracle against the LIVE reference and writes tests/golden/*.pt.

Run in the build container only (needs /root/reference, which does not exist on
the GPU box):   python -m oracle.make_golden
The reference is imported unmodified through an import shim (stubs for the four
training-only dependencies that are not installed here; T5Config.from_pretrained
patched so that no network is touched) -- SURVEY.md section 8c.

What is checked at generation time (hard asserts):
  * oracle.unet_ref.unet_forward == reference Unet.forward (cond and null branch)
  * oracle.sampler_ref.imagen_sample == reference Imagen.sample on the same seed
  * oracle.sampler_ref.elucidated_sample == reference ElucidatedImagen.sample
  * cascade (lowres_cond SR unet, memory_efficient) variants of the above
What is written: small fixtures (weights of tiny U-Nets + inputs + reference
outputs) that the CPU and GPU test-suites replay without the reference.
"""
from __future__ import annotations

import os
import sys
import types
import importlib.machinery

import torch


def _install_shim():
    import transformers  # noqa: F401  (must be imported before the stubs)

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__spec__ = importlib.machinery.ModuleSpec(name, None)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    class _Any:
        def __init__(self, *a, **k):
            pass

    k = stub('kornia')
    k.augmentation = stub('kornia.augmentation', RandomCrop=_Any)
    stub('accelerate', Accelerator=_Any, DistributedType=_Any, DistributedDataParallelKwargs=_Any)
    stub('ema_pytorch', EMA=_Any)
    stub('pytorch_warmup', LinearWarmup=_Any)
    from transformers import T5Config
    T5Config.from_pretrained = classmethod(
        lambda cls, name, *a, **kw: T5Config(d_model=1024 if 'large' in name else 768))
    sys.path.insert(0, '/root/reference')


def _maxdiff(a, b):
    return (a - b).abs().max().item()


def main():
    _install_shim()
    import imagen_pytorch as ref
    from oracle import unet_ref, sampler_ref

    out_dir = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
    os.makedirs(out_dir, exist_ok=True)
    torch.set_num_threads(8)

    # ---------------------------------------------------------------- 1. base unet forward (cfg-1 shape family)
    shapes_out = {}

    def build(name, kwargs, seed, lowres=False):
        u = ref.Unet(**kwargs, lowres_cond=lowres)
        shapes = {k: tuple(v.shape) for k, v in u.state_dict().items()}
        shapes_out[name] = shapes
        sd = unet_ref.synth_state_dict(shapes, seed=seed)
        u.load_state_dict(sd)                       # strict: every key, every shape
        u.eval()
        cfg = unet_ref.unet_config(**kwargs, lowres_cond=lowres)
        return u, sd, cfg

    base_kw = dict(dim=32, dim_mults=(1, 2, 4, 8), text_embed_dim=64, max_text_len=24)
    u, sd, cfg = build('base', base_kw, 0)
    g = torch.Generator().manual_seed(7)
    B = 2
    x = torch.randn(B, 3, 32, 32, generator=g)
    t = torch.tensor([-1.7, 0.6])
    te = torch.randn(B, 24, 64, generator=g)
    te[1, 17:] = 0.                                   # ragged text -> mask has False entries
    tm = torch.any(te != 0., dim=-1)
    with torch.no_grad():
        r_c = u(x, t, text_embeds=te, text_mask=tm)
        r_n = u(x, t, text_embeds=te, text_mask=tm, cond_drop_prob=1.)
        r_g = u.forward_with_cond_scale(x, t, text_embeds=te, text_mask=tm, cond_scale=3.)
        o_c = unet_ref.unet_forward(sd, cfg, x, t, text_embeds=te, text_mask=tm)
        o_n = unet_ref.unet_forward(sd, cfg, x, t, text_embeds=te, text_mask=tm, cond_drop_prob=1.)
        o_g = unet_ref.unet_forward_with_cond_scale(sd, cfg, x, t, text_embeds=te, text_mask=tm, cond_scale=3.)
    for name, a, b in (('cond', r_c, o_c), ('null', r_n, o_n), ('cfg', r_g, o_g)):
        d = _maxdiff(a, b)
        print(f'[unet base {name}] ref-vs-oracle max|d| = {d:.3e}  (|ref|max {a.abs().max():.3f})')
        assert d < 1e-5 * max(1., a.abs().max().item()), name   # fp32 re-association only
    torch.save(dict(kwargs=base_kw, wseed=0, x=x, t=t, text_embeds=te, text_mask=tm,
                    out_cond=r_c, out_null=r_n, out_cfg3=r_g), os.path.join(out_dir, 'unet_base_dim32.pt'))

    # ---------------------------------------------------------------- 2. SR unet forward (lowres_cond, memory_efficient, mixed attns)
    sr_kw = dict(dim=32, dim_mults=(1, 2, 4), text_embed_dim=64, max_text_len=24, num_resnet_blocks=(1, 2, 2),
                 layer_attns=(False, False, True), layer_cross_attns=(False, False, True), memory_efficient=True)
    us, sds, cfgs = build('sr', sr_kw, 3, lowres=True)
    xs = torch.randn(B, 3, 32, 32, generator=g)
    low = torch.randn(B, 3, 32, 32, generator=g)
    lnt = torch.tensor([0.7093, 0.7093])
    with torch.no_grad():
        rs = us(xs, t, text_embeds=te, text_mask=tm, lowres_cond_img=low, lowres_noise_times=lnt)
        os_ = unet_ref.unet_forward(sds, cfgs, xs, t, text_embeds=te, text_mask=tm, lowres_cond_img=low, lowres_noise_times=lnt)
    d = _maxdiff(rs, os_)
    print(f'[unet sr] ref-vs-oracle max|d| = {d:.3e}')
    assert d < 1e-5 * max(1., rs.abs().max().item())
    torch.save(dict(kwargs=sr_kw, wseed=3, x=xs, t=t, text_embeds=te, text_mask=tm, lowres_cond_img=low,
                    lowres_noise_times=lnt, out=rs), os.path.join(out_dir, 'unet_sr_dim32.pt'))

    # ---------------------------------------------------------------- 3. DDPM sample trajectory (base, CFG)
    imagen = ref.Imagen(unets=u, image_sizes=32, timesteps=6, text_embed_dim=64)
    imagen.unets[0].load_state_dict(sd)
    torch.manual_seed(11)
    r_img = imagen.sample(text_embeds=te, cond_scale=3., use_tqdm=False)
    torch.manual_seed(11)
    trace = []
    o_img = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=te, timesteps=6, cond_scale=3., trace=trace)
    d = _maxdiff(r_img, o_img)
    print(f'[ddpm sample] ref-vs-oracle max|d| = {d:.3e}')
    assert d < 1e-4
    torch.save(dict(kwargs=base_kw, wseed=0, text_embeds=te, seed=11, timesteps=6, cond_scale=3.,
                    out=r_img, trace=torch.stack(trace)), os.path.join(out_dir, 'ddpm_sample_dim32.pt'))

    # ---------------------------------------------------------------- 4. cascade DDPM sample (base 16 -> SR 32)
    imagen2 = ref.Imagen(unets=(ref.Unet(**base_kw), ref.Unet(**sr_kw)), image_sizes=(16, 32), timesteps=3, text_embed_dim=64)
    imagen2.unets[0].load_state_dict(sd)
    imagen2.unets[1].load_state_dict(sds)
    torch.manual_seed(5)
    r_c2 = imagen2.sample(text_embeds=te, cond_scale=2., use_tqdm=False, return_all_unet_outputs=True)
    torch.manual_seed(5)
    o_c2 = sampler_ref.imagen_sample([(sd, cfg), (sds, cfgs)], (16, 32), text_embeds=te, timesteps=3, cond_scale=2.,
                                     return_all_unet_outputs=True)
    for a, b in zip(r_c2, o_c2):
        d = _maxdiff(a, b)
        print(f'[ddpm cascade {tuple(a.shape)}] ref-vs-oracle max|d| = {d:.3e}')
        assert d < 1e-4
    torch.save(dict(base_kwargs=base_kw, sr_kwargs=sr_kw, wseed_base=0, wseed_sr=3, text_embeds=te, seed=5, timesteps=3,
                    cond_scale=2., outs=[o.clone() for o in r_c2]), os.path.join(out_dir, 'ddpm_cascade_dim32.pt'))

    # ---------------------------------------------------------------- 5. Elucidated sample (base + cascade)
    el = ref.ElucidatedImagen(unets=(ref.Unet(**base_kw), ref.Unet(**sr_kw)), image_sizes=(16, 32), text_embed_dim=64,
                              num_sample_steps=4)
    el.unets[0].load_state_dict(sd)
    el.unets[1].load_state_dict(sds)
    torch.manual_seed(9)
    r_e = el.sample(text_embeds=te, cond_scale=2., use_tqdm=False)
    torch.manual_seed(9)
    o_e = sampler_ref.elucidated_sample([(sd, cfg), (sds, cfgs)], (16, 32), text_embeds=te, cond_scale=2.,
                                        hparams=dict(num_sample_steps=4))
    d = _maxdiff(r_e, o_e)
    print(f'[edm cascade] ref-vs-oracle max|d| = {d:.3e}')
    # sigma_max=80 puts |x| ~ 80 in fp32 (1 ulp = 7.6e-6) and the untrained net amplifies it
    # over 7 Heun evals x 2 stages: measured 7.6e-6 after 2 steps, ~5e-5 after 4, 2.3e-4 here.
    assert d < 1e-3
    torch.save(dict(base_kwargs=base_kw, sr_kwargs=sr_kw, wseed_base=0, wseed_sr=3, text_embeds=te, seed=9,
                    num_sample_steps=4, cond_scale=2., out=r_e), os.path.join(out_dir, 'edm_cascade_dim32.pt'))

    # ---------------------------------------------------------------- 5b. sampler options on the DDPM loop (SURVEY.md 8f.2)
    # init image + skipped steps, and RePaint inpainting (resample 3x), on the cascade so both the per-stage resize of the
    # init / inpaint images and the low-res hand-off are covered
    g2 = torch.Generator().manual_seed(21)
    init_img = torch.rand(B, 3, 32, 32, generator=g2)
    inp_img = torch.rand(B, 3, 32, 32, generator=g2)
    inp_mask = torch.zeros(B, 32, 32, dtype=torch.bool)
    inp_mask[0, 8:24, 4:20] = True
    inp_mask[1, :, 16:] = True
    imagen3 = ref.Imagen(unets=(ref.Unet(**base_kw), ref.Unet(**sr_kw)), image_sizes=(16, 32), timesteps=4, text_embed_dim=64)
    imagen3.unets[0].load_state_dict(sd)
    imagen3.unets[1].load_state_dict(sds)
    torch.manual_seed(13)
    r_is = imagen3.sample(text_embeds=te, cond_scale=2., use_tqdm=False, init_images=init_img, skip_steps=1, return_all_unet_outputs=True)
    torch.manual_seed(13)
    o_is = sampler_ref.imagen_sample([(sd, cfg), (sds, cfgs)], (16, 32), text_embeds=te, timesteps=4, cond_scale=2.,
                                     init_images=init_img, skip_steps=1, return_all_unet_outputs=True)
    for a, b in zip(r_is, o_is):
        d = _maxdiff(a, b)
        print(f'[ddpm init+skip {tuple(a.shape)}] ref-vs-oracle max|d| = {d:.3e}')
        assert d < 1e-4
    torch.manual_seed(17)
    r_ip = imagen3.sample(text_embeds=te, cond_scale=2., use_tqdm=False, inpaint_images=inp_img, inpaint_masks=inp_mask,
                          inpaint_resample_times=3, return_all_unet_outputs=True)
    torch.manual_seed(17)
    o_ip = sampler_ref.imagen_sample([(sd, cfg), (sds, cfgs)], (16, 32), text_embeds=te, timesteps=4, cond_scale=2.,
                                     inpaint_images=inp_img, inpaint_masks=inp_mask, inpaint_resample_times=3,
                                     return_all_unet_outputs=True)
    for a, b in zip(r_ip, o_ip):
        d = _maxdiff(a, b)
        print(f'[ddpm inpaint {tuple(a.shape)}] ref-vs-oracle max|d| = {d:.3e}')
        assert d < 1e-4
    torch.save(dict(base_kwargs=base_kw, sr_kwargs=sr_kw, wseed_base=0, wseed_sr=3, text_embeds=te, timesteps=4, cond_scale=2.,
                    init_images=init_img, skip_steps=1, seed_init=13, outs_init=[o.clone() for o in r_is],
                    inpaint_images=inp_img, inpaint_masks=inp_mask, inpaint_resample_times=3, seed_inpaint=17,
                    outs_inpaint=[o.clone() for o in r_ip]), os.path.join(out_dir, 'ddpm_options_dim32.pt'))

    # ---------------------------------------------------------------- 5c. the same options on the EDM loop
    # sigma_max = 2 instead of 80: with the default the untrained nets amplify fp32 re-association noise to 5e-2 over the extra
    # resampling evaluations (the oracle differs that much from ITSELF between 1 and 8 threads), which would pin nothing
    el3 = ref.ElucidatedImagen(unets=(ref.Unet(**base_kw), ref.Unet(**sr_kw)), image_sizes=(16, 32), text_embed_dim=64, num_sample_steps=3,
                               sigma_max=2.)
    el3.unets[0].load_state_dict(sd)
    el3.unets[1].load_state_dict(sds)
    torch.manual_seed(23)
    r_eis = el3.sample(text_embeds=te, cond_scale=2., use_tqdm=False, init_images=init_img, skip_steps=1, return_all_unet_outputs=True)
    torch.manual_seed(23)
    o_eis = sampler_ref.elucidated_sample([(sd, cfg), (sds, cfgs)], (16, 32), text_embeds=te, cond_scale=2.,
                                          hparams=dict(num_sample_steps=3, sigma_max=2.), init_images=init_img, skip_steps=1,
                                          return_all_unet_outputs=True)
    for a, b in zip(r_eis, o_eis):
        d = _maxdiff(a, b)
        print(f'[edm init+skip {tuple(a.shape)}] ref-vs-oracle max|d| = {d:.3e}')
        assert d < 1e-4
    torch.manual_seed(29)
    r_eip = el3.sample(text_embeds=te, cond_scale=2., use_tqdm=False, inpaint_images=inp_img, inpaint_masks=inp_mask,
                       inpaint_resample_times=2, return_all_unet_outputs=True)
    torch.manual_seed(29)
    o_eip = sampler_ref.elucidated_sample([(sd, cfg), (sds, cfgs)], (16, 32), text_embeds=te, cond_scale=2.,
                                          hparams=dict(num_sample_steps=3, sigma_max=2.), inpaint_images=inp_img, inpaint_masks=inp_mask,
                                          inpaint_resample_times=2, return_all_unet_outputs=True)
    for a, b in zip(r_eip, o_eip):
        d = _maxdiff(a, b)
        print(f'[edm inpaint {tuple(a.shape)}] ref-vs-oracle max|d| = {d:.3e}')
        # the SR stage amplifies the 1.6e-5 hand-off difference ~40x even at sigma_max = 2 (untrained net, 2 x 2 x 3 evaluations);
        # the test-suites compare trajectories statistically (mean |d| < 1e-2), so 2e-3 max still pins the control flow
        assert d < 2e-3
    torch.save(dict(base_kwargs=base_kw, sr_kwargs=sr_kw, wseed_base=0, wseed_sr=3, text_embeds=te, num_sample_steps=3, sigma_max=2., cond_scale=2.,
                    init_images=init_img, skip_steps=1, seed_init=23, outs_init=[o.clone() for o in r_eis],
                    inpaint_images=inp_img, inpaint_masks=inp_mask, inpaint_resample_times=2, seed_inpaint=29,
                    outs_inpaint=[o.clone() for o in r_eip]), os.path.join(out_dir, 'edm_options_dim32.pt'))

    # ---------------------------------------------------------------- 5d. self-conditioning (Unet(self_cond=True), imagen_pytorch.py:1541-1543, :2252)
    sc_kw = dict(base_kw, self_cond=True)
    usc, sdsc, cfgsc = build('selfcond', sc_kw, 5)
    xsc = torch.randn(B, 3, 32, 32, generator=g)
    scin = torch.randn(B, 3, 32, 32, generator=g).clamp(-1, 1)
    with torch.no_grad():
        r_sc = usc(xsc, t, text_embeds=te, text_mask=tm, self_cond=scin)
        r_sc0 = usc(xsc, t, text_embeds=te, text_mask=tm)                       # no self_cond given: zeros
        o_sc = unet_ref.unet_forward(sdsc, cfgsc, xsc, t, text_embeds=te, text_mask=tm, self_cond=scin)
        o_sc0 = unet_ref.unet_forward(sdsc, cfgsc, xsc, t, text_embeds=te, text_mask=tm)
    for name, a, b in (('given', r_sc, o_sc), ('zeros', r_sc0, o_sc0)):
        d = _maxdiff(a, b)
        print(f'[unet self_cond {name}] ref-vs-oracle max|d| = {d:.3e}')
        assert d < 1e-5 * max(1., a.abs().max().item())
    im_sc = ref.Imagen(unets=ref.Unet(**sc_kw), image_sizes=32, timesteps=4, text_embed_dim=64)
    im_sc.unets[0].load_state_dict(sdsc)
    torch.manual_seed(53)
    r_scs = im_sc.sample(text_embeds=te, cond_scale=2., use_tqdm=False)
    torch.manual_seed(53)
    o_scs = sampler_ref.imagen_sample([(sdsc, cfgsc)], (32,), text_embeds=te, timesteps=4, cond_scale=2.)
    d = _maxdiff(r_scs, o_scs)
    print(f'[ddpm self_cond sample] ref-vs-oracle max|d| = {d:.3e}')
    assert d < 1e-4
    el_sc = ref.ElucidatedImagen(unets=ref.Unet(**sc_kw), image_sizes=32, text_embed_dim=64, num_sample_steps=3, sigma_max=2.)
    el_sc.unets[0].load_state_dict(sdsc)
    torch.manual_seed(59)
    r_sce = el_sc.sample(text_embeds=te, cond_scale=2., use_tqdm=False)
    torch.manual_seed(59)
    o_sce = sampler_ref.elucidated_sample([(sdsc, cfgsc)], (32,), text_embeds=te, cond_scale=2., hparams=dict(num_sample_steps=3, sigma_max=2.))
    d = _maxdiff(r_sce, o_sce)
    print(f'[edm self_cond sample] ref-vs-oracle max|d| = {d:.3e}')
    assert d < 1e-4
    torch.save(dict(kwargs=sc_kw, wseed=5, x=xsc, t=t, text_embeds=te, text_mask=tm, self_cond=scin, out=r_sc, out_zeros=r_sc0,
                    timesteps=4, cond_scale=2., seed_ddpm=53, out_ddpm=r_scs, num_sample_steps=3, sigma_max=2., seed_edm=59, out_edm=r_sce),
               os.path.join(out_dir, 'self_cond_dim32.pt'))

    # ---------------------------------------------------------------- 5e. pred_objectives 'v' / 'x_start' (imagen_pytorch.py:2085-2090, :308-312)
    obj = {}
    for objective, seed in (('v', 71), ('x_start', 73)):
        im_o = ref.Imagen(unets=ref.Unet(**base_kw), image_sizes=32, timesteps=4, text_embed_dim=64, pred_objectives=objective)
        im_o.unets[0].load_state_dict(sd)
        torch.manual_seed(seed)
        r_o = im_o.sample(text_embeds=te, cond_scale=2., use_tqdm=False)
        torch.manual_seed(seed)
        o_o = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=te, timesteps=4, cond_scale=2., pred_objectives=objective)
        d = _maxdiff(r_o, o_o)
        print(f'[ddpm objective {objective}] ref-vs-oracle max|d| = {d:.3e}')
        assert d < 1e-4
        obj[objective] = dict(seed=seed, out=r_o)
    torch.save(dict(kwargs=base_kw, wseed=0, text_embeds=te, timesteps=4, cond_scale=2., objectives=obj),
               os.path.join(out_dir, 'ddpm_objectives_dim32.pt'))

    # ---------------------------------------------------------------- 5f. BASELINE.json shapes: the oracle pinned against the live reference
    # (i) configs[1] architecture: Unet(dim=128) @64x64 with (256, 768) text embeddings -- cond / null / CFG-3 forward.
    # Inputs and weights are rebuilt from seeds in the tests (synth_state_dict over the key->shape contract), only outputs are stored.
    def seeded_inputs(seed, B, size, L=256, D=768, ragged=True):
        gg = torch.Generator().manual_seed(seed)
        x_ = torch.randn(B, 3, size, size, generator=gg)
        te_ = torch.randn(B, L, D, generator=gg)
        if ragged and B > 1:
            te_[1, L // 3:] = 0.
        return x_, te_, torch.any(te_ != 0., dim=-1)

    big = {}
    for name, kw, wseed, iseed in (('dim128', dict(dim=128), 11, 101), ('dim192', dict(dim=192), 12, 102)):
        ub, sdb, cfgb = build('base_' + name, kw, wseed)
        Bb = 2 if name == 'dim128' else 1
        xb, teb, tmb = seeded_inputs(iseed, Bb, 64)
        tb = torch.tensor([0.8, -1.3])[:Bb]
        with torch.no_grad():
            r1 = ub(xb, tb, text_embeds=teb, text_mask=tmb)
            o1 = unet_ref.unet_forward(sdb, cfgb, xb, tb, text_embeds=teb, text_mask=tmb)
            entry = dict(kwargs=kw, wseed=wseed, iseed=iseed, B=Bb, t=tb, out_cond=r1)
            d = _maxdiff(r1, o1)
            print(f'[unet {name} @64 cond] ref-vs-oracle max|d| = {d:.3e}  (|ref|max {r1.abs().max():.3f})')
            assert d < 2e-5 * max(1., r1.abs().max().item())
            if name == 'dim128':
                r0 = ub(xb, tb, text_embeds=teb, text_mask=tmb, cond_drop_prob=1.)
                o0 = unet_ref.unet_forward(sdb, cfgb, xb, tb, text_embeds=teb, text_mask=tmb, cond_drop_prob=1.)
                d = _maxdiff(r0, o0)
                print(f'[unet {name} @64 null] ref-vs-oracle max|d| = {d:.3e}')
                assert d < 2e-5 * max(1., r0.abs().max().item())
                entry.update(out_null=r0, out_cfg3=r0 + (r1 - r0) * 3.)
        big[name] = entry
        del ub, sdb
    # (ii) configs[3] second stage: SRUnet256(lowres_cond=True) forward at 256 x 256, B = 1
    torch.manual_seed(0)
    usr = ref.SRUnet256(lowres_cond=True)
    shp = {k: tuple(v.shape) for k, v in usr.state_dict().items()}
    sdsr = unet_ref.synth_state_dict(shp, seed=13)
    usr.load_state_dict(sdsr)
    usr.eval()
    sr256_kw = dict(dim=128, dim_mults=(1, 2, 4, 8), num_resnet_blocks=(2, 4, 8, 8), layer_attns=(False, False, False, True),
                    layer_cross_attns=(False, False, False, True), attn_heads=8, ff_mult=2., memory_efficient=True)
    cfgsr = unet_ref.unet_config(**sr256_kw, lowres_cond=True)
    xr, ter, tmr = seeded_inputs(103, 1, 256)
    lowr = torch.randn(1, 3, 256, 256, generator=torch.Generator().manual_seed(104))
    with torch.no_grad():
        rr = usr(xr, torch.tensor([0.4]), text_embeds=ter, text_mask=tmr, lowres_cond_img=lowr, lowres_noise_times=torch.tensor([0.7093]))
        orr = unet_ref.unet_forward(sdsr, cfgsr, xr, torch.tensor([0.4]), text_embeds=ter, text_mask=tmr, lowres_cond_img=lowr,
                                    lowres_noise_times=torch.tensor([0.7093]))
    d = _maxdiff(rr, orr)
    print(f'[SRUnet256 @256] ref-vs-oracle max|d| = {d:.3e}  (|ref|max {rr.abs().max():.3f})')
    assert d < 2e-5 * max(1., rr.abs().max().item())
    big['srunet256'] = dict(kwargs=sr256_kw, wseed=13, iseed=103, lseed=104, t=torch.tensor([0.4]), lowres_noise_times=torch.tensor([0.7093]), out=rr)
    del usr, sdsr
    # (iii) SURVEY.md 8f.1: the SRUnet1024 architecture through the upscale-only entry (start_at_unet_number = 2) at 64 -> 128
    sr1024_kw = dict(dim=128, dim_mults=(1, 2, 4, 8), num_resnet_blocks=(2, 4, 8, 8), layer_attns=False,
                     layer_cross_attns=(False, False, False, True), attn_heads=8, ff_mult=2., memory_efficient=True)
    torch.manual_seed(0)
    u1k = ref.SRUnet1024()
    im1k = ref.Imagen(unets=(ref.Unet(**base_kw), u1k), image_sizes=(64, 128), timesteps=3, text_embed_dim=64)
    shp1k = {k: tuple(v.shape) for k, v in im1k.unets[1].state_dict().items()}
    sd1k = unet_ref.synth_state_dict(shp1k, seed=14)
    im1k.unets[1].load_state_dict(sd1k)
    cfg1k = unet_ref.unet_config(**sr1024_kw, lowres_cond=True, text_embed_dim=64)
    start = torch.rand(B, 3, 64, 64, generator=torch.Generator().manual_seed(105))
    torch.manual_seed(79)
    r1k = im1k.sample(text_embeds=te, cond_scale=2., use_tqdm=False, start_at_unet_number=2, start_image_or_video=start)
    torch.manual_seed(79)
    o1k = sampler_ref.imagen_sample([(sd, cfg), (sd1k, cfg1k)], (64, 128), text_embeds=te, timesteps=3, cond_scale=2.,
                                    start_at_unet_number=2, start_image=start)
    d = _maxdiff(r1k, o1k)
    print(f'[SRUnet1024 arch, upscale-only 64->128] ref-vs-oracle max|d| = {d:.3e}')
    assert d < 1e-4
    big['srunet1024_upscale'] = dict(kwargs=sr1024_kw, wseed=14, text_embeds=te, start_seed=105, seed=79, timesteps=3, cond_scale=2., out=r1k)
    shapes_out['srunet1024_t64'] = shp1k
    # (iv) BASELINE.json configs[0]: base Unet dim=32 dim_mults=(1,2,4,8) @64x64, bs=2, 50 DDPM steps, text (256, 768), reference p_sample_loop
    kw0 = dict(dim=32, dim_mults=(1, 2, 4, 8))
    u0, sd0, cfg0 = build('base_dim32_full', kw0, 15)
    x0_, te0, _ = seeded_inputs(106, 2, 64)
    im0 = ref.Imagen(unets=ref.Unet(**kw0), image_sizes=64, timesteps=50)
    im0.unets[0].load_state_dict(sd0)
    torch.manual_seed(83)
    r50 = im0.sample(text_embeds=te0, cond_scale=1., use_tqdm=False)
    torch.manual_seed(83)
    o50 = sampler_ref.imagen_sample([(sd0, cfg0)], (64,), text_embeds=te0, timesteps=50, cond_scale=1.)
    d = _maxdiff(r50, o50)
    print(f'[configs[0]: dim32 @64, bs 2, 50 DDPM steps] ref-vs-oracle max|d| = {d:.3e}')
    assert d < 1e-3
    big['cfg0_50steps'] = dict(kwargs=kw0, wseed=15, iseed=106, seed=83, timesteps=50, out=r50)
    # the 256 x 256 output in a file of its own keeps every fixture under 1 MB
    torch.save(big.pop('srunet256'), os.path.join(out_dir, 'baseline_srunet256.pt'))
    torch.save(big, os.path.join(out_dir, 'baseline_shapes.pt'))

    # ---------------------------------------------------------------- 5g. boundary options: attn_dim_head = 32 (the reference's UnetConfig default,
    # configs.py:49-50) with attn_heads = 4, and cond_images (imagen_pytorch.py:1553-1560) -- forward + a 3-step CFG DDPM sample
    dh_kw = dict(dim=32, dim_mults=(1, 2, 4), text_embed_dim=64, max_text_len=24, attn_dim_head=32, attn_heads=4, cond_images_channels=3)
    udh, sddh, cfgdh = build('dh32_cond', dh_kw, 17)
    gdh = torch.Generator().manual_seed(107)
    xdh = torch.randn(B, 3, 32, 32, generator=gdh)
    cimg = torch.rand(B, 3, 16, 16, generator=gdh)                  # half resolution: resized (nearest) inside the U-Net
    with torch.no_grad():
        r_dh = udh(xdh, t, text_embeds=te, text_mask=tm, cond_images=cimg)
        r_dh0 = udh(xdh, t, text_embeds=te, text_mask=tm, cond_images=cimg, cond_drop_prob=1.)
        o_dh = unet_ref.unet_forward(sddh, cfgdh, xdh, t, text_embeds=te, text_mask=tm, cond_images=cimg)
        o_dh0 = unet_ref.unet_forward(sddh, cfgdh, xdh, t, text_embeds=te, text_mask=tm, cond_images=cimg, cond_drop_prob=1.)
    for name, a, b in (('cond', r_dh, o_dh), ('null', r_dh0, o_dh0)):
        d = _maxdiff(a, b)
        print(f'[unet dim_head 32 + cond_images {name}] ref-vs-oracle max|d| = {d:.3e}')
        assert d < 1e-5 * max(1., a.abs().max().item())
    im_dh = ref.Imagen(unets=ref.Unet(**dh_kw), image_sizes=32, timesteps=3, text_embed_dim=64)
    im_dh.unets[0].load_state_dict(sddh)
    torch.manual_seed(89)
    r_dhs = im_dh.sample(text_embeds=te, cond_images=cimg, cond_scale=2., use_tqdm=False)
    torch.manual_seed(89)
    o_dhs = sampler_ref.imagen_sample([(sddh, cfgdh)], (32,), text_embeds=te, timesteps=3, cond_scale=2., cond_images=cimg)
    d = _maxdiff(r_dhs, o_dhs)
    print(f'[ddpm dim_head 32 + cond_images sample] ref-vs-oracle max|d| = {d:.3e}')
    assert d < 1e-4
    torch.save(dict(kwargs=dh_kw, wseed=17, x=xdh, t=t, text_embeds=te, text_mask=tm, cond_images=cimg, out_cond=r_dh, out_null=r_dh0,
                    timesteps=3, cond_scale=2., seed=89, out_sample=r_dhs), os.path.join(out_dir, 'unet_dh32_cond_dim32.pt'))

    # ---------------------------------------------------------------- 6. schedule / scalar known answers
    tt = torch.tensor([1., .75, .5, .25, 0., 0.2])
    torch.save(dict(t=tt, cosine=ref.imagen_pytorch.alpha_cosine_log_snr(tt), linear=ref.imagen_pytorch.beta_linear_log_snr(tt),
                    edm_sigmas=el.sample_schedule(4, 7, 0.002, 80)), os.path.join(out_dir, 'schedules.pt'))

    # ---------------------------------------------------------------- 7. state_dict key/shape contract of the default configs
    contract = {'test_base': shapes_out['base'], 'test_sr': shapes_out['sr'], 'test_selfcond': shapes_out['selfcond'],
                'base_dim192': shapes_out['base_dim192'], 'srunet1024_t64': shapes_out['srunet1024_t64'], 'test_dh32_cond': shapes_out['dh32_cond']}
    for name, kw in (('base_dim128', dict(dim=128)), ('base_dim32', dict(dim=32, dim_mults=(1, 2, 4, 8)))):
        torch.manual_seed(0)
        m = ref.Unet(**kw)
        contract[name] = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    torch.manual_seed(0)
    m = ref.SRUnet256(lowres_cond=True)
    contract['srunet256'] = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    torch.save(contract, os.path.join(out_dir, 'state_dict_contract.pt'))
    print('golden fixtures written to', out_dir)
    for f in sorted(os.listdir(out_dir)):
        print('  ', f, os.path.getsize(os.path.join(out_dir, f)) // 1024, 'KiB')


if __name__ == '__main__':
    main()
