"""CPU: the oracle (oracle/) reproduces the golden vectors generated from the live reference
(oracle/make_golden.py).  These fixtures are the reference's outputs, not the oracle's."""
import torch

from oracle import unet_ref, sampler_ref
from tests.helpers import load_golden, synth_weights

torch.set_num_threads(max(1, min(8, torch.get_num_threads())))


def test_unet_base_forward_matches_reference_golden():
    g = load_golden('unet_base_dim32.pt')
    sd = synth_weights('test_base', g['wseed'])
    cfg = unet_ref.unet_config(**g['kwargs'])
    kw = dict(text_embeds=g['text_embeds'], text_mask=g['text_mask'])
    with torch.no_grad():
        out = unet_ref.unet_forward(sd, cfg, g['x'], g['t'], **kw)
        out_null = unet_ref.unet_forward(sd, cfg, g['x'], g['t'], cond_drop_prob=1., **kw)
    assert out.abs().max() > 1.0                       # not the vacuous zero-init case
    assert (out - g['out_cond']).abs().max() < 1e-4
    assert (out_null - g['out_null']).abs().max() < 1e-4
    assert (out - out_null).abs().max() > 0.1          # text conditioning actually matters


def test_unet_sr_forward_matches_reference_golden():
    g = load_golden('unet_sr_dim32.pt')
    sd = synth_weights('test_sr', g['wseed'])
    cfg = unet_ref.unet_config(**g['kwargs'], lowres_cond=True)
    with torch.no_grad():
        out = unet_ref.unet_forward(sd, cfg, g['x'], g['t'], text_embeds=g['text_embeds'], text_mask=g['text_mask'],
                                    lowres_cond_img=g['lowres_cond_img'], lowres_noise_times=g['lowres_noise_times'])
    assert (out - g['out']).abs().max() < 1e-4


def test_ddpm_sample_matches_reference_golden():
    g = load_golden('ddpm_sample_dim32.pt')
    sd = synth_weights('test_base', g['wseed'])
    cfg = unet_ref.unet_config(**g['kwargs'])
    torch.manual_seed(g['seed'])
    trace = []
    with torch.no_grad():
        out = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=g['text_embeds'], timesteps=g['timesteps'],
                                        cond_scale=g['cond_scale'], trace=trace)
    assert (out - g['out']).abs().max() < 1e-4
    assert (torch.stack(trace) - g['trace']).abs().max() < 1e-3
    assert 0. <= out.min() and out.max() <= 1.


def test_ddpm_cascade_matches_reference_golden():
    g = load_golden('ddpm_cascade_dim32.pt')
    sdb, sds = synth_weights('test_base', g['wseed_base']), synth_weights('test_sr', g['wseed_sr'])
    cb = unet_ref.unet_config(**g['base_kwargs'])
    cs = unet_ref.unet_config(**g['sr_kwargs'], lowres_cond=True)
    torch.manual_seed(g['seed'])
    with torch.no_grad():
        outs = sampler_ref.imagen_sample([(sdb, cb), (sds, cs)], (16, 32), text_embeds=g['text_embeds'], timesteps=g['timesteps'],
                                         cond_scale=g['cond_scale'], return_all_unet_outputs=True)
    for o, r in zip(outs, g['outs']):
        assert (o - r).abs().max() < 1e-4


def test_edm_cascade_matches_reference_golden():
    g = load_golden('edm_cascade_dim32.pt')
    sdb, sds = synth_weights('test_base', g['wseed_base']), synth_weights('test_sr', g['wseed_sr'])
    cb = unet_ref.unet_config(**g['base_kwargs'])
    cs = unet_ref.unet_config(**g['sr_kwargs'], lowres_cond=True)
    torch.manual_seed(g['seed'])
    with torch.no_grad():
        out = sampler_ref.elucidated_sample([(sdb, cb), (sds, cs)], (16, 32), text_embeds=g['text_embeds'], cond_scale=g['cond_scale'],
                                            hparams=dict(num_sample_steps=g['num_sample_steps']))
    # sigma_max = 80 puts |x| ~ 80 in fp32; the untrained net amplifies 1-ulp re-association differences (see make_golden.py)
    assert (out - g['out']).abs().max() < 2e-3


def _cascade_models(g):
    sdb, sds = synth_weights('test_base', g['wseed_base']), synth_weights('test_sr', g['wseed_sr'])
    return [(sdb, unet_ref.unet_config(**g['base_kwargs'])), (sds, unet_ref.unet_config(**g['sr_kwargs'], lowres_cond=True))]


def test_ddpm_sampler_options_match_reference_golden():
    """init_images + skip_steps and RePaint inpainting on the DDPM cascade (imagen_pytorch.py:2205-2279), SURVEY.md 8f.2."""
    g = load_golden('ddpm_options_dim32.pt')
    models = _cascade_models(g)
    common = dict(text_embeds=g['text_embeds'], timesteps=g['timesteps'], cond_scale=g['cond_scale'], return_all_unet_outputs=True)
    with torch.no_grad():
        torch.manual_seed(g['seed_init'])
        a = sampler_ref.imagen_sample(models, (16, 32), init_images=g['init_images'], skip_steps=g['skip_steps'], **common)
        torch.manual_seed(g['seed_inpaint'])
        b = sampler_ref.imagen_sample(models, (16, 32), inpaint_images=g['inpaint_images'], inpaint_masks=g['inpaint_masks'],
                                      inpaint_resample_times=g['inpaint_resample_times'], **common)
    for o, r in zip(a + b, g['outs_init'] + g['outs_inpaint']):
        assert (o - r).abs().max() < 1e-4
    # masked pixels of the final image are the known image, bit for bit (:2285-2288)
    m = g['inpaint_masks'][:, None].expand(-1, 3, -1, -1)
    assert torch.equal(b[1][m], ((g['inpaint_images'] * 2 - 1 + 1) * 0.5)[m])


def test_edm_sampler_options_match_reference_golden():
    """The same options on ElucidatedImagen.one_unet_sample (elucidated_imagen.py:446-447, :455-462, :476-477, :498-499, :533-542)."""
    g = load_golden('edm_options_dim32.pt')
    models = _cascade_models(g)
    common = dict(text_embeds=g['text_embeds'], cond_scale=g['cond_scale'], return_all_unet_outputs=True,
                  hparams=dict(num_sample_steps=g['num_sample_steps'], sigma_max=g['sigma_max']))
    with torch.no_grad():
        torch.manual_seed(g['seed_init'])
        a = sampler_ref.elucidated_sample(models, (16, 32), init_images=g['init_images'], skip_steps=g['skip_steps'], **common)
        torch.manual_seed(g['seed_inpaint'])
        b = sampler_ref.elucidated_sample(models, (16, 32), inpaint_images=g['inpaint_images'], inpaint_masks=g['inpaint_masks'],
                                          inpaint_resample_times=g['inpaint_resample_times'], **common)
    for o, r in zip(a, g['outs_init']):
        assert (o - r).abs().max() < 1e-4
    for o, r in zip(b, g['outs_inpaint']):
        assert (o - r).abs().max() < 5e-3      # the SR stage amplifies fp32 re-association noise (see make_golden.py)
    m = g['inpaint_masks'][:, None].expand(-1, 3, -1, -1)
    assert torch.equal(b[1][m], ((g['inpaint_images'] * 2 - 1 + 1) * 0.5)[m])


def test_self_conditioning_matches_reference_golden():
    """Unet(self_cond=True): forward with a given / default (zeros) self_cond, and both samplers feeding x_start back
    (imagen_pytorch.py:1541-1543, :2252; elucidated_imagen.py:496, :518, :538)."""
    g = load_golden('self_cond_dim32.pt')
    sd, cfg = synth_weights('test_selfcond', g['wseed']), unet_ref.unet_config(**g['kwargs'])
    kw = dict(text_embeds=g['text_embeds'], text_mask=g['text_mask'])
    with torch.no_grad():
        a = unet_ref.unet_forward(sd, cfg, g['x'], g['t'], self_cond=g['self_cond'], **kw)
        b = unet_ref.unet_forward(sd, cfg, g['x'], g['t'], **kw)
        torch.manual_seed(g['seed_ddpm'])
        c = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=g['text_embeds'], timesteps=g['timesteps'], cond_scale=g['cond_scale'])
        torch.manual_seed(g['seed_edm'])
        d = sampler_ref.elucidated_sample([(sd, cfg)], (32,), text_embeds=g['text_embeds'], cond_scale=g['cond_scale'],
                                          hparams=dict(num_sample_steps=g['num_sample_steps'], sigma_max=g['sigma_max']))
    assert (a - g['out']).abs().max() < 1e-4 and (b - g['out_zeros']).abs().max() < 1e-4
    assert (a - b).abs().max() > 1e-2                      # the self-conditioning channels matter
    assert (c - g['out_ddpm']).abs().max() < 1e-4 and (d - g['out_edm']).abs().max() < 1e-3


def test_schedule_known_answers():
    g = load_golden('schedules.pt')
    assert torch.allclose(sampler_ref.alpha_cosine_log_snr(g['t']), g['cosine'], atol=1e-6)
    assert torch.allclose(sampler_ref.beta_linear_log_snr(g['t']), g['linear'], atol=1e-6)
    assert torch.allclose(sampler_ref.edm_sample_schedule(4, 7, 0.002, 80), g['edm_sigmas'], rtol=1e-6)
    # SURVEY.md appendix A.2 / A.3 probe values
    assert abs(sampler_ref.alpha_cosine_log_snr(torch.tensor([0.5])).item() + 0.0249) < 1e-3
    assert abs(sampler_ref.beta_linear_log_snr(torch.tensor([0.2])).item() - 0.7093) < 1e-3
    assert abs(sampler_ref.edm_sample_schedule(4, 7, 0.002, 80)[1].item() - 9.7232) < 1e-2


def test_pred_objectives_v_and_x_start_match_reference_golden():
    """pred_objective 'v' / 'x_start' (imagen_pytorch.py:2085-2090, :308-312) of the oracle's DDPM loop against the live reference."""
    g = load_golden('ddpm_objectives_dim32.pt')
    sd = synth_weights('test_base', g['wseed'])
    cfg = unet_ref.unet_config(**g['kwargs'])
    outs = {}
    for objective, e in g['objectives'].items():
        torch.manual_seed(e['seed'])
        with torch.no_grad():
            outs[objective] = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=g['text_embeds'], timesteps=g['timesteps'],
                                                        cond_scale=g['cond_scale'], pred_objectives=objective)
        assert (outs[objective] - e['out']).abs().max() < 1e-4
    assert (outs['v'] - outs['x_start']).abs().mean() > 1e-2      # two different parameterisations, two different images


def test_baseline_shape_fixture_is_complete():
    """tests/golden/baseline_shapes.pt and baseline_srunet256.pt hold the live reference's outputs at the BASELINE.json shapes (the
    GPU suite replays them); here: the fixture's entries and the key->shape contracts they rebuild their weights from."""
    from tests.helpers import contract
    g, c = load_golden('baseline_shapes.pt'), contract()
    assert set(g) == {'dim128', 'dim192', 'srunet1024_upscale', 'cfg0_50steps'}
    g['srunet256'] = load_golden('baseline_srunet256.pt')
    assert g['dim128']['out_cond'].shape == (2, 3, 64, 64) and g['dim192']['out_cond'].shape == (1, 3, 64, 64)
    assert g['srunet256']['out'].shape == (1, 3, 256, 256) and g['srunet1024_upscale']['out'].shape == (2, 3, 128, 128)
    assert g['cfg0_50steps']['out'].shape == (2, 3, 64, 64) and g['cfg0_50steps']['timesteps'] == 50
    for name in ('base_dim128', 'base_dim192', 'base_dim32', 'srunet256', 'srunet1024_t64'):
        assert name in c and len(c[name]) > 100
    assert torch.allclose(g['dim128']['out_cfg3'], g['dim128']['out_null'] + (g['dim128']['out_cond'] - g['dim128']['out_null']) * 3.)


def test_dim_head_32_and_cond_images_match_reference_golden():
    """attn_dim_head = 32 / attn_heads = 4 (the reference's UnetConfig default head width) + cond_images (imagen_pytorch.py:1553-1560)."""
    g = load_golden('unet_dh32_cond_dim32.pt')
    sd = synth_weights('test_dh32_cond', g['wseed'])
    cfg = unet_ref.unet_config(**g['kwargs'])
    kw = dict(text_embeds=g['text_embeds'], text_mask=g['text_mask'], cond_images=g['cond_images'])
    with torch.no_grad():
        out = unet_ref.unet_forward(sd, cfg, g['x'], g['t'], **kw)
        out0 = unet_ref.unet_forward(sd, cfg, g['x'], g['t'], cond_drop_prob=1., **kw)
    assert (out - g['out_cond']).abs().max() < 1e-4 and (out0 - g['out_null']).abs().max() < 1e-4
    torch.manual_seed(g['seed'])
    with torch.no_grad():
        img = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=g['text_embeds'], timesteps=g['timesteps'], cond_scale=g['cond_scale'],
                                        cond_images=g['cond_images'])
    assert (img - g['out_sample']).abs().max() < 1e-4
