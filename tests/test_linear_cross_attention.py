"""Unet(use_linear_cross_attn=...): LinearCrossAttention (imagen_pytorch.py:836-874) on the B200 path.

CPU: the parameter layout and the oracle against the live-reference fixture tests/golden/linear_cross_attn_dim32.pt, and the launch plan.
GPU (-m gpu): the two kernels against torch fp32, whole forwards against the reference outputs, a DDPM trajectory against the oracle on
the same noise, graph == eager, batched CFG == separate passes, and one forward at the BASELINE.json cfg-2 shape.
Measured errors are recorded in the same parity report as tests/test_gpu_unet.py's values."""
import pytest
import torch

import imagen_pytorch_b200 as b2
from imagen_pytorch_b200 import _lib
from imagen_pytorch_b200.params import UnetArch, param_table
from oracle import unet_ref, sampler_ref
from oracle.linear_cross_ref import linear_layers
from tests.helpers import load_golden, rel_err, seeded_inputs, shapes_of
from tests.test_gpu_unet import record as _record

DEV = 'cuda'
G = load_golden('linear_cross_attn_dim32.pt')
CASES = list(G['cases'])


def record(name, **vals):
    _record('linear_cross_' + name, **vals)


def _model(name):
    kw = G['cases'][name]
    sd = unet_ref.synth_state_dict(G['contracts'][name], seed=G['outs'][name]['wseed'])
    return kw, sd, unet_ref.unet_config(**kw)


def _args(kw, dev='cpu'):
    a = dict(text_embeds=G['text_embeds'], text_mask=G['text_mask']) if kw.get('cond_on_text', True) else {}
    if kw.get('lowres_cond'):
        a.update(lowres_cond_img=G['lowres_cond_img'], lowres_noise_times=G['lowres_noise_times'])
    return {k: v.to(dev) for k, v in a.items()}


# ------------------------------------------------------------------------------------------------ CPU

@pytest.mark.parametrize('name', CASES)
def test_param_table_matches_reference_contract(name):
    mine = {k: tuple(v[0]) for k, v in param_table(UnetArch(**G['cases'][name])).items()}
    assert mine == {k: tuple(v) for k, v in G['contracts'][name].items()}


def test_level_flags():
    a = UnetArch(**G['cases']['A'])
    assert [(a.down_level(i)['cross'], a.down_level(i)['linear_cross']) for i in range(3)] == [(True, True), (True, False), (True, True)]
    assert [a.up_level(i)['linear_cross'] for i in range(3)] == [True, False, True]      # up levels run in reverse order
    assert not any(UnetArch(dim=32, dim_mults=(1, 2)).down_level(i)['linear_cross'] for i in range(2))


@pytest.mark.parametrize('name', CASES)
def test_oracle_matches_reference_golden(name):
    kw, sd, cfg = _model(name)
    ref = G['outs'][name]
    x, t = G['x'], G['t']
    with torch.no_grad(), linear_layers(cfg):
        got = dict(cond=unet_ref.unet_forward(sd, cfg, x, t, **_args(kw)))
        if 'null' in ref:
            got['null'] = unet_ref.unet_forward(sd, cfg, x, t, cond_drop_prob=1., **_args(kw))
            got['cfg3'] = unet_ref.unet_forward_with_cond_scale(sd, cfg, x, t, cond_scale=3., **_args(kw))
    for k, v in got.items():
        assert (v - ref[k]).abs().max().item() < 1e-5 * max(1., ref[k].abs().max().item()), k   # fp32 re-association only


def test_oracle_sample_matches_reference_golden():
    kw, sd, cfg = _model('A')
    s = G['sample']
    torch.manual_seed(s['seed'])
    with torch.no_grad(), linear_layers(cfg):
        out = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=G['text_embeds'], timesteps=s['timesteps'], cond_scale=s['cond_scale'])
    assert (out - s['out']).abs().max().item() < 1e-4


def test_plan_compiles_on_the_meta_device():
    """Case A: 4 linear cross-attention layers (levels 0 and 2, down and up), each one context kernel + one attention kernel;
    level 1 and the two mid blocks keep b200_attention, as do the level-2 transformers and the mid attention."""
    from imagen_pytorch_b200.unet import UnetPlan
    plan = UnetPlan(b2.Unet(**G['cases']['A']), 4, 2, 32, 32, 6, torch.device('meta'))
    names = [o[2] for o in plan._ops]
    assert names.count('b200_linear_xattn_context') == 4 and names.count('b200_linear_cross_attention') == 4
    assert names.count('b200_attention') == 3 + 4
    assert plan.n_launches == 134
    # every context kernel runs after the per-step time-row refresh of its K/V buffers
    assert names.index('b200_update_time_rows') < names.index('b200_linear_xattn_context')
    assert sum(L['linear'] for L in plan.cross_layers) == 4 and len(plan.cross_layers) == 4 + 2 + 2


def test_tuple_flag_of_wrong_length_is_rejected():
    with pytest.raises(AssertionError):
        UnetArch(dim=32, dim_mults=(1, 2, 4), use_linear_cross_attn=(True, False))


# ------------------------------------------------------------------------------------------------ GPU: kernels vs torch fp32

def _bf(t):
    return t.to(torch.bfloat16)


def _torch_linear_xattn(q, k, v, heads, dh):
    """fp32 reference on the bf16-rounded operands: q [R, n, heads*64], k / v [R, nk, heads*64] -> [R, n, heads, dh]."""
    R, n, _ = q.shape
    qf, kf, vf = (t.float().view(t.shape[0], t.shape[1], heads, 64)[..., :dh] for t in (q, k, v))
    qs = qf.softmax(dim=-1) * 8
    ks = kf.softmax(dim=1)
    ctx = torch.einsum('rjhd,rjhe->rhde', ks, vf)
    return torch.einsum('rnhd,rhde->rnhe', qs, ctx)


@pytest.mark.gpu
@pytest.mark.parametrize('heads,dh', [(8, 64), (4, 32)], ids=['8x64', '4x32pad'])
@pytest.mark.parametrize('nk', [3, 27, 39, 64])
def test_kernels_match_torch_fp32(heads, dh, nk):
    """q and k scaled x20: without a max subtraction in either softmax the exponentials overflow to inf / NaN.  Channels dh..63 of a
    padded head hold large values too: they must take no part in the softmax over d (their outputs are not compared: to_out's
    padded weight columns are zero)."""
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator(device=DEV).manual_seed(1000 * heads + nk)
    worst = 0.
    for R in (1, 5):
        for n in (9, 64, 1600, 4096):
            inner = heads * 64
            q = _bf(torch.randn(R, n, inner, device=DEV, generator=gen) * 20)
            k = _bf(torch.randn(R, nk, inner, device=DEV, generator=gen) * 20)
            v = _bf(torch.randn(R, nk, inner, device=DEV, generator=gen))
            ctx = torch.empty(R, heads, 64, 64, dtype=torch.bfloat16, device=DEV)
            o = torch.full((R, n, inner), float('nan'), dtype=torch.bfloat16, device=DEV)
            _lib.check(lib.b200_linear_xattn_context(k.data_ptr(), v.data_ptr(), nk * inner, inner, nk, R, heads, dh, ctx.data_ptr(), st),
                       'b200_linear_xattn_context')
            _lib.check(lib.b200_linear_cross_attention(q.data_ptr(), o.data_ptr(), n * inner, inner, n, ctx.data_ptr(), R, heads, dh, st),
                       'b200_linear_cross_attention')
            torch.cuda.synchronize()
            ref = _torch_linear_xattn(q, k, v, heads, dh)
            got = o.float().view(R, n, heads, 64)[..., :dh]
            assert torch.isfinite(got).all(), (R, n)
            e = rel_err(got, ref)
            worst = max(worst, e)
            assert e < 1.5e-2, (R, n, e)      # P, C and O are rounded to bf16 (2^-9 each)
            if dh < 64:
                assert (ctx.float()[:, :, dh:, :] == 0).all()       # C rows of padded channels are exact zeros
    record(f'kernel_{heads}x{dh}_keys{nk}', worst_rel_l2=worst)


# ------------------------------------------------------------------------------------------------ GPU: whole path

def _unet(name, impl=_lib.IMPL_TCGEN05):
    kw, sd, cfg = _model(name)
    u = b2.Unet(**kw)
    u.load_state_dict(sd)
    u._gemm_impl = impl
    return u.to(DEV), sd, cfg


@pytest.mark.gpu
@pytest.mark.parametrize('impl', [_lib.IMPL_TCGEN05, _lib.IMPL_SIMT_CHECKER], ids=['tcgen05', 'simt'])
@pytest.mark.parametrize('name', CASES)
def test_forward_matches_reference_golden(name, impl):
    u, _, _ = _unet(name, impl)
    kw, ref = G['cases'][name], G['outs'][name]
    x, t, args = G['x'].to(DEV), G['t'].to(DEV), _args(kw, DEV)
    got = dict(cond=u(x, t, **args))
    if 'null' in ref:
        got['null'] = u(x, t, cond_drop_prob=1., **args)
        got['cfg3'] = u.forward_with_cond_scale(x, t, cond_scale=3., **args)
    errs = {k: rel_err(v, ref[k]) for k, v in got.items()}
    record(f'forward_{name}_impl{impl}', **errs)
    assert all(e < 3e-2 for e in errs.values()), errs


@pytest.mark.gpu
def test_ddpm_sample_matches_oracle_with_shared_noise():
    u, sd, cfg = _unet('A')
    s, te = G['sample'], G['text_embeds']
    im = b2.Imagen(u, image_sizes=32, timesteps=s['timesteps'], text_embed_dim=64).to(DEV)
    torch.manual_seed(131)
    out = im.sample(text_embeds=te.to(DEV), cond_scale=s['cond_scale'], use_tqdm=False)
    torch.manual_seed(131)
    with torch.no_grad(), linear_layers(cfg):
        ref = sampler_ref.imagen_sample([(sd, cfg)], (32,), text_embeds=te, timesteps=s['timesteps'], cond_scale=s['cond_scale'],
                                        randn=lambda shape: torch.randn(tuple(shape), device=DEV).cpu())
    d = (out.cpu() - ref).abs()
    record('ddpm_sample_A_6steps', mean_abs=d.mean(), max_abs=d.max())
    assert out.shape == ref.shape and d.mean() < 1e-2


@pytest.mark.gpu
def test_graph_equals_eager_and_batched_cfg_equals_separate_passes(monkeypatch):
    u, _, _ = _unet('A')
    te = G['text_embeds'].to(DEV)
    im = b2.Imagen(u, image_sizes=32, timesteps=5, text_embed_dim=64).to(DEV)
    torch.manual_seed(5)
    a = im.sample(text_embeds=te, cond_scale=2., use_tqdm=False)
    n_graph = im.last_launch_count
    monkeypatch.setenv('B200_IMAGEN_NO_GRAPH', '1')
    torch.manual_seed(5)
    b = im.sample(text_embeds=te, cond_scale=2., use_tqdm=False)
    assert torch.equal(a, b)
    assert n_graph == 5 * (u.plan(4, 2, 32, 32, 5).n_launches + 2)
    x, t, args = G['x'].to(DEV), G['t'].to(DEV), _args(G['cases']['A'], DEV)
    cond, null = u(x, t, **args), u(x, t, cond_drop_prob=1., **args)
    cfg = u.forward_with_cond_scale(x, t, cond_scale=3., **args)
    assert torch.allclose(cfg, null + (cond - null) * 3., rtol=0, atol=1e-5)


@pytest.mark.gpu
def test_baseline_shape_forward_matches_oracle_dim128_64px():
    """Unet(dim=128, use_linear_cross_attn=True) @64x64, B = 2, text (2, 256, 768) with a ragged mask: every level's cross-attention
    is linear (4096 / 1024 / 256 / 64 pixels per sample).  The oracle runs in fp32 on the GPU (TF32 off)."""
    kw = dict(dim=128, use_linear_cross_attn=True)
    u = b2.Unet(**kw)
    shapes = shapes_of(u)
    sd = unet_ref.synth_state_dict(shapes, seed=11)
    u.load_state_dict(sd)
    u = u.to(DEV)
    x, te, tm = (v.to(DEV) for v in seeded_inputs(101, 2, 64))
    t = torch.tensor([0.8, -1.3], device=DEV)
    out = u(x, t, text_embeds=te, text_mask=tm)
    sdg = {k: v.to(DEV) for k, v in sd.items()}
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        cfg = unet_ref.unet_config(**kw)
        with torch.no_grad(), linear_layers(cfg):
            ref = unet_ref.unet_forward(sdg, cfg, x, t, text_embeds=te, text_mask=tm)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    e = rel_err(out, ref)
    d = (out - ref).abs()
    record('baseline_dim128_64px', rel_l2=e, max_abs=d.max(), ref_max=ref.abs().max())
    assert torch.isfinite(out).all() and e < 3e-2
