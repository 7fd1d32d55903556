"""GPU (-m gpu): parity at the BASELINE.json shapes (VERDICT r01 "next round" item 1).

Single forwards are compared with outputs of the LIVE reference (tests/golden/baseline_*.pt, written by
oracle/make_golden.py, which also hard-asserts oracle == reference on the same inputs); inputs and weights are rebuilt
from seeds.  Trajectories are compared with the oracle run on this box's host cores on the SAME CUDA-drawn noise.
Tolerances: bf16 activations / fp32 accumulation against an fp32 reference, see DESIGN.md section 4; the measured
numbers land in gpurun_out/parity_report_baseline.json (committed as profiles/r02_parity_report.json)."""
import json
import os

import pytest
import torch

import imagen_pytorch_b200 as b2
from oracle import unet_ref, sampler_ref
from tests.helpers import load_golden, contract, rel_err, seeded_inputs, shapes_of

pytestmark = pytest.mark.gpu
DEV = 'cuda'
REPORT = {}


def record(name, **vals):
    REPORT[name] = {k: float(v) for k, v in vals.items()}
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gpurun_out')
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, 'parity_report_baseline.json'), 'w') as f:
        json.dump(REPORT, f, indent=1)


def cuda_randn(shape):
    return torch.randn(tuple(shape), device=DEV).cpu()


def stats(out, ref):
    d = (out.float().cpu() - ref.float().cpu()).abs()
    return dict(rel_l2=rel_err(out, ref), mean_abs=d.mean().item(), max_abs=d.max().item(), ref_max=ref.abs().max().item())


def image_stats(out, ref):
    d = (out.float().cpu() - ref.float().cpu()).abs()
    return dict(mean_abs=d.mean().item(), max_abs=d.max().item(), psnr=(-10 * torch.log10((d ** 2).mean())).item())


def load_unet(cls_or_kwargs, shapes, wseed, **extra):
    u = cls_or_kwargs(**extra) if callable(cls_or_kwargs) else b2.Unet(**cls_or_kwargs, **extra)
    assert shapes_of(u) == {k: tuple(v) for k, v in shapes.items()}, 'state_dict layout differs from the reference contract'
    sd = unet_ref.synth_state_dict(shapes, seed=wseed)
    u.load_state_dict(sd)
    return u.to(DEV), sd


# ------------------------------------------------------------------------------------------------ single forwards vs the live reference

def test_cfg2_unet_dim128_64px_forward_matches_reference():
    """BASELINE.json configs[1] architecture: Unet(dim=128) @64x64, text (2, 256, 768) with a ragged mask: N = 4096 self-attention
    inside the real network, 256-token -> 36-latent perceiver, K up to 13824 convs.  cond / null / CFG-3."""
    g = load_golden('baseline_shapes.pt')['dim128']
    u, _ = load_unet(g['kwargs'], contract()['base_dim128'], g['wseed'])
    x, te, tm = seeded_inputs(g['iseed'], g['B'], 64)
    x, te, tm, t = x.to(DEV), te.to(DEV), tm.to(DEV), g['t'].to(DEV)
    out = u(x, t, text_embeds=te, text_mask=tm)
    null = u(x, t, text_embeds=te, text_mask=tm, cond_drop_prob=1.)
    cfg = u.forward_with_cond_scale(x, t, text_embeds=te, text_mask=tm, cond_scale=3.)
    s_c, s_n, s_g = stats(out, g['out_cond']), stats(null, g['out_null']), stats(cfg, g['out_cfg3'])
    record('cfg2_dim128_forward', cond=s_c['rel_l2'], null=s_n['rel_l2'], cfg3=s_g['rel_l2'], cond_max_abs=s_c['max_abs'],
           cfg3_max_abs=s_g['max_abs'], ref_max=s_c['ref_max'])
    assert s_c['rel_l2'] < 3e-2 and s_n['rel_l2'] < 3e-2 and s_g['rel_l2'] < 5e-2
    assert s_c['max_abs'] < 0.1 * max(1.0, s_c['ref_max'])


def test_cfg5_unet_dim192_forward_matches_reference():
    """BASELINE.json configs[4] architecture: Unet(dim=192) @64x64 (2304-channel concat norms, 1536-wide deepest level)."""
    g = load_golden('baseline_shapes.pt')['dim192']
    u, _ = load_unet(g['kwargs'], contract()['base_dim192'], g['wseed'])
    x, te, tm = seeded_inputs(g['iseed'], g['B'], 64)
    out = u(x.to(DEV), g['t'].to(DEV), text_embeds=te.to(DEV), text_mask=tm.to(DEV))
    s = stats(out, g['out_cond'])
    record('cfg5_dim192_forward', **s)
    assert s['rel_l2'] < 3e-2 and s['max_abs'] < 0.1 * max(1.0, s['ref_max'])


def test_cfg4_srunet256_forward_256px_matches_reference():
    """BASELINE.json configs[3] second stage: SRUnet256(lowres_cond=True) at 256 x 256, B = 1 (memory_efficient, 64 Ki pixel rows)."""
    g = load_golden('baseline_srunet256.pt')
    u, _ = load_unet(b2.SRUnet256, contract()['srunet256'], g['wseed'], lowres_cond=True)
    x, te, tm = seeded_inputs(g['iseed'], 1, 256)
    low = torch.randn(1, 3, 256, 256, generator=torch.Generator().manual_seed(g['lseed']))
    out = u(x.to(DEV), g['t'].to(DEV), text_embeds=te.to(DEV), text_mask=tm.to(DEV), lowres_cond_img=low.to(DEV),
            lowres_noise_times=g['lowres_noise_times'].to(DEV))
    s = stats(out, g['out'])
    record('cfg4_srunet256_forward_256px', **s)
    assert s['rel_l2'] < 3e-2 and s['max_abs'] < 0.1 * max(1.0, s['ref_max'])


# ------------------------------------------------------------------------------------------------ trajectories vs the oracle (shared noise)

def test_cfg1_dim32_64px_50_ddpm_steps_matches_oracle():
    """BASELINE.json configs[0] exactly: base Unet dim=32 dim_mults=(1,2,4,8) @64x64, bs=2, 50 DDPM steps, text (256, 768),
    cond_scale 1 -- the full-length trajectory (bf16 drift over 50 stochastic, dynamically thresholded steps)."""
    g = load_golden('baseline_shapes.pt')['cfg0_50steps']
    u, sd = load_unet(g['kwargs'], contract()['base_dim32'], g['wseed'])
    _, te, _ = seeded_inputs(g['iseed'], 2, 64)
    im = b2.Imagen(u, image_sizes=64, timesteps=g['timesteps']).to(DEV)
    torch.manual_seed(321)
    out = im.sample(text_embeds=te.to(DEV), cond_scale=1., use_tqdm=False)
    torch.manual_seed(321)
    with torch.no_grad():
        ref = sampler_ref.imagen_sample([(sd, unet_ref.unet_config(**g['kwargs']))], (64,), text_embeds=te, timesteps=g['timesteps'],
                                        cond_scale=1., randn=cuda_randn)
    s = image_stats(out, ref)
    record('cfg1_dim32_64px_50steps', **s)
    assert out.shape == (2, 3, 64, 64) and 0 <= out.min() and out.max() <= 1
    assert s['mean_abs'] < 2e-2 and s['psnr'] > 28.0


@pytest.mark.parametrize('objective', ['v', 'x_start'])
def test_pred_objectives_match_oracle(objective):
    """pred_objective 'v' / 'x_start' (imagen_pytorch.py:2085-2090, :308-312): the step kernel's objective switch."""
    g = load_golden('ddpm_objectives_dim32.pt')
    from tests.helpers import synth_weights
    sd = synth_weights('test_base', g['wseed'])
    u = b2.Unet(**g['kwargs'])
    u.load_state_dict(sd)
    im = b2.Imagen(u.to(DEV), image_sizes=32, timesteps=g['timesteps'], text_embed_dim=64, pred_objectives=objective).to(DEV)
    te = g['text_embeds']
    torch.manual_seed(5)
    out = im.sample(text_embeds=te.to(DEV), cond_scale=g['cond_scale'], use_tqdm=False)
    torch.manual_seed(5)
    with torch.no_grad():
        ref = sampler_ref.imagen_sample([(sd, unet_ref.unet_config(**g['kwargs']))], (32,), text_embeds=te, timesteps=g['timesteps'],
                                        cond_scale=g['cond_scale'], pred_objectives=objective, randn=cuda_randn)
        ref_noise = sampler_ref.imagen_sample([(sd, unet_ref.unet_config(**g['kwargs']))], (32,), text_embeds=te, timesteps=g['timesteps'],
                                              cond_scale=g['cond_scale'], pred_objectives='noise',
                                              randn=lambda s, _g=torch.Generator().manual_seed(0): torch.randn(tuple(s), generator=_g))
    s = image_stats(out, ref)
    record(f'ddpm_objective_{objective}', **s)
    assert s['mean_abs'] < 1e-2 and s['max_abs'] < 0.1
    assert (ref - ref_noise).abs().mean() > 1e-2            # the objective switch is live in the oracle (a different image than 'noise')


def test_srunet1024_architecture_upscale_only_matches_oracle():
    """SURVEY.md 8f.1: the conv-only SRUnet1024 stage (imagen_pytorch.py:1771-1783) through start_at_unet_number = 2 /
    start_image_or_video (:2396-2403) at 64 -> 128, against the oracle on the same noise."""
    g = load_golden('baseline_shapes.pt')['srunet1024_upscale']
    gb = load_golden('unet_base_dim32.pt')
    first = b2.Unet(**gb['kwargs'])                          # stage 1 is never planned or run
    sr = b2.SRUnet1024(lowres_cond=True, text_embed_dim=64)
    shapes = contract()['srunet1024_t64']
    assert shapes_of(sr) == {k: tuple(v) for k, v in shapes.items()}
    sd = unet_ref.synth_state_dict(shapes, seed=g['wseed'])
    sr.load_state_dict(sd)
    im = b2.Imagen((first, sr), image_sizes=(64, 128), timesteps=g['timesteps'], text_embed_dim=64).to(DEV)
    assert im.unets[1] is sr
    te = g['text_embeds']
    start = torch.rand(2, 3, 64, 64, generator=torch.Generator().manual_seed(g['start_seed']))
    torch.manual_seed(77)
    out = im.sample(text_embeds=te.to(DEV), cond_scale=g['cond_scale'], use_tqdm=False, start_at_unet_number=2, start_image_or_video=start.to(DEV))
    cfg = unet_ref.unet_config(**g['kwargs'], lowres_cond=True, text_embed_dim=64)
    torch.manual_seed(77)
    with torch.no_grad():
        ref = sampler_ref.imagen_sample([(None, None), (sd, cfg)], (64, 128), text_embeds=te, timesteps=g['timesteps'], cond_scale=g['cond_scale'],
                                        start_at_unet_number=2, start_image=start, randn=cuda_randn)
    s = image_stats(out, ref)
    record('srunet1024_arch_upscale_64_128', **s)
    assert out.shape == (2, 3, 128, 128) and s['mean_abs'] < 1e-2 and s['max_abs'] < 0.15


# ------------------------------------------------------------------------------------------------ boundary options (VERDICT r01 item 9)

def test_dim_head_32_and_cond_images_forward_and_sample():
    """Unet(attn_dim_head=32, attn_heads=4, cond_images_channels=3): heads zero-padded to the kernels' 64-wide head layout
    (params.pad_attention_heads), conditioning image as a fourth stem source (b200_im2col_init4) -- forward against the live
    reference's golden, 3-step CFG DDPM sample against the oracle on the same noise."""
    from tests.helpers import synth_weights
    g = load_golden('unet_dh32_cond_dim32.pt')
    sd = synth_weights('test_dh32_cond', g['wseed'])
    u = b2.Unet(**g['kwargs'])
    u.load_state_dict(sd)
    u = u.to(DEV)
    kw = dict(text_embeds=g['text_embeds'].to(DEV), text_mask=g['text_mask'].to(DEV), cond_images=g['cond_images'].to(DEV))
    out = u(g['x'].to(DEV), g['t'].to(DEV), **kw)
    out0 = u(g['x'].to(DEV), g['t'].to(DEV), cond_drop_prob=1., **kw)
    e, e0 = rel_err(out, g['out_cond']), rel_err(out0, g['out_null'])
    im = b2.Imagen(u, image_sizes=32, timesteps=g['timesteps'], text_embed_dim=64).to(DEV)
    torch.manual_seed(3)
    img = im.sample(text_embeds=g['text_embeds'].to(DEV), cond_images=g['cond_images'].to(DEV), cond_scale=g['cond_scale'], use_tqdm=False)
    torch.manual_seed(3)
    with torch.no_grad():
        ref = sampler_ref.imagen_sample([(sd, unet_ref.unet_config(**g['kwargs']))], (32,), text_embeds=g['text_embeds'], timesteps=g['timesteps'],
                                        cond_scale=g['cond_scale'], cond_images=g['cond_images'], randn=cuda_randn)
    s = image_stats(img, ref)
    record('dim_head32_cond_images', fwd_cond=e, fwd_null=e0, **s)
    assert e < 3e-2 and e0 < 3e-2 and s['mean_abs'] < 1e-2
    with pytest.raises(AssertionError):                     # cond image required once the U-Net was built with cond_images_channels (:1555)
        im.sample(text_embeds=g['text_embeds'].to(DEV), cond_scale=1., use_tqdm=False)


# ------------------------------------------------------------------------------------------------ callers either side of the path (SURVEY.md 8f.3 / 8f.4)

def test_sample_from_texts_and_trainer_checkpoint_with_ema():
    """sample(texts=...) through the encode_text hook equals sample(text_embeds=...) of the same encoder output; a TrainedSampler loaded
    from an ImagenTrainer.save-layout checkpoint samples with the EMA weights (chunked by max_batch_size) unless use_non_ema."""
    from tests.helpers import synth_weights
    from tests.test_host_logic import _ToyTokenizer, _toy_t5
    from imagen_pytorch_b200 import t5, TrainedSampler
    g = load_golden('unet_base_dim32.pt')
    sd_online, sd_ema = synth_weights('test_base', 1), synth_weights('test_base', 2)
    t5.register_text_encoder('toy-t5', _toy_t5(), _ToyTokenizer())

    def imagen_with(sd):
        u = b2.Unet(**g['kwargs'])
        u.load_state_dict(sd)
        return b2.Imagen(u.to(DEV), image_sizes=32, timesteps=3, text_encoder_name='toy-t5').to(DEV)

    im = imagen_with(sd_online)
    assert im.text_embed_dim == 64
    texts = ['a cat', 'a dog on a skateboard', 'nothing']
    torch.manual_seed(11)
    a = im.sample(texts=texts, cond_scale=2., use_tqdm=False)
    emb, mask = t5.t5_encode_text(texts, name='toy-t5', return_attn_mask=True)
    torch.manual_seed(11)
    b = im.sample(text_embeds=emb, text_masks=mask, cond_scale=2., use_tqdm=False)
    assert a.shape == (3, 3, 32, 32) and torch.equal(a, b)
    ckpt = dict(model={'unets.0.' + k: v for k, v in sd_online.items()}, ema={'0.ema_model.' + k: v for k, v in sd_ema.items()}, version='1.26.2',
                steps=torch.tensor([3]))
    ts = TrainedSampler(imagen_with(synth_weights('test_base', 3)))
    ts.load(ckpt)
    torch.manual_seed(12)
    e = ts.sample(text_embeds=emb[:2], text_masks=mask[:2], cond_scale=2., use_tqdm=False)
    torch.manual_seed(12)
    e_ref = imagen_with(sd_ema).sample(text_embeds=emb[:2], text_masks=mask[:2], cond_scale=2., use_tqdm=False)
    torch.manual_seed(12)
    o = ts.sample(text_embeds=emb[:2], text_masks=mask[:2], cond_scale=2., use_tqdm=False, use_non_ema=True)
    torch.manual_seed(12)
    o_ref = imagen_with(sd_online).sample(text_embeds=emb[:2], text_masks=mask[:2], cond_scale=2., use_tqdm=False)
    assert torch.equal(e, e_ref) and torch.equal(o, o_ref) and not torch.equal(e, o)
    # chunked sampling: two chunks of (2, 1) samples, each chunk drawing its own noise in order
    torch.manual_seed(13)
    c = ts.sample(text_embeds=emb, text_masks=mask, cond_scale=2., use_tqdm=False, max_batch_size=2)
    torch.manual_seed(13)
    c0 = ts.sample(text_embeds=emb[:2], text_masks=mask[:2], cond_scale=2., use_tqdm=False)
    c1 = ts.sample(text_embeds=emb[2:], text_masks=mask[2:], cond_scale=2., use_tqdm=False)
    assert c.shape[0] == 3 and torch.equal(c, torch.cat((c0, c1)))


# ------------------------------------------------------------------------------------------------ plan cache (ADVICE r01)

def test_plan_and_step_graph_are_reused_across_sample_calls_and_track_weight_updates():
    """sample() twice on the same Imagen: the second call must reuse the UnetPlan and the captured step graph (no rebuild inside
    reset_unets_all_one_device) and still give what a fresh model gives; an in-place weight update / a parent load_state_dict
    must invalidate the packed weights."""
    g = load_golden('ddpm_sample_dim32.pt')
    from tests.helpers import synth_weights
    sd = synth_weights('test_base', g['wseed'])

    def fresh():
        u = b2.Unet(**g['kwargs'])
        u.load_state_dict(sd)
        return b2.Imagen(u.to(DEV), image_sizes=32, timesteps=4, text_embed_dim=64).to(DEV)

    te1 = g['text_embeds'].to(DEV)
    te2 = torch.randn_like(te1)
    im = fresh()
    torch.manual_seed(1)
    a1 = im.sample(text_embeds=te1, cond_scale=2., use_tqdm=False)
    u = im.unets[0]
    plans = dict(u._plans)
    plan = next(iter(plans.values()))
    graphs = dict(plan.sampler_state['ddpm']['graphs'])
    assert len(plans) == 1 and len(graphs) == 1
    torch.manual_seed(2)
    a2 = im.sample(text_embeds=te2, cond_scale=2., use_tqdm=False)
    assert dict(u._plans) == plans and next(iter(u._plans.values())) is plan
    assert plan.sampler_state['ddpm']['graphs'] == graphs   # same captured graph object replayed
    torch.manual_seed(2)
    b2_ = fresh().sample(text_embeds=te2, cond_scale=2., use_tqdm=False)
    assert torch.equal(a2, b2_) and not torch.equal(a1, a2)
    # parent-module load_state_dict with different weights -> the plan is rebuilt and the output follows the new weights
    sd_new = {k: v * 1.05 if v.ndim > 1 else v for k, v in sd.items()}
    im.load_state_dict({'unets.0.' + k: v for k, v in sd_new.items()}, strict=False)
    torch.manual_seed(2)
    a3 = im.sample(text_embeds=te2, cond_scale=2., use_tqdm=False)
    assert next(iter(u._plans.values())) is not plan
    u2 = b2.Unet(**g['kwargs'])
    u2.load_state_dict(sd_new)
    torch.manual_seed(2)
    b3 = b2.Imagen(u2.to(DEV), image_sizes=32, timesteps=4, text_embed_dim=64).to(DEV).sample(text_embeds=te2, cond_scale=2., use_tqdm=False)
    assert torch.equal(a3, b3) and not torch.equal(a3, a2)
