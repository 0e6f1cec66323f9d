"""GPU tests of several ControlNets and ControlNet guess mode on the fused denoising loop: tiny and SD-1.5-size loops
against the fp32 oracle loop (oracle/controlnet_multi.py `loop_controlnet_multi`), the pipeline `__call__` against the
reference's own `__call__` (tests/golden/pipeline_controlnet_multi_call.npz), exact identities of the residual sum, the
standalone guess-mode forward, and the plan cache.

Tolerances are those of tests/test_pipelines_gpu.py (trajectories: rel-L2 <= 5e-2, cosine >= 0.998; SD-1.5 size
cosine >= 0.999) and tests/test_nets_gpu.py (single forward: rel-L2 <= 3e-2)."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
DEV = "cuda"


def _rel(a, b):
    return ((a.float() - b.float()).norm() / (b.float().norm() + 1e-12)).item()


def _cos(a, b):
    return torch.nn.functional.cosine_similarity(a.float().flatten(), b.float().flatten(), dim=0).item()


@pytest.fixture(scope="module", autouse=True)
def _fp32_exact():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


def _net(kind, cin, seed, tiny=True):
    """(fp32 oracle on the GPU, product model) with the same synthetic weights"""
    from oracle.unet import ControlNetOracle, UNet2DConditionOracle, UNetConfig
    from powerpaint_b200.engine import NetConfig
    from powerpaint_b200.models import ControlNetModel, UNet2DConditionModel, synthetic_state_dict

    o = UNetConfig.tiny(cin) if tiny else UNetConfig.sd15(cin)
    n = NetConfig(in_channels=cin, block_out_channels=o.block_out_channels, attention_head_dim=o.attention_head_dim,
                  cross_attention_dim=o.cross_attention_dim, norm_num_groups=o.norm_num_groups)
    sd = synthetic_state_dict(n, kind, seed)
    om = {"unet": UNet2DConditionOracle, "controlnet": ControlNetOracle}[kind](o)
    om.load_state_dict(sd)
    pm = {"unet": UNet2DConditionModel, "controlnet": ControlNetModel}[kind].from_state_dict(n, sd).to(DEV)
    return om.to(DEV).eval(), pm, o


def _scheds(steps, total=50):
    from oracle.ddim import DDIMOracle
    from powerpaint_b200.schedulers import DDIMScheduler

    so, sp = DDIMOracle(), DDIMScheduler()
    so.set_timesteps(total)
    sp.set_timesteps(total)
    so.timesteps = so.timesteps[:steps]
    return so, sp, sp.timesteps[:steps]


def _report(name, **kv):
    print(name, kv)


def _inputs(B, h, cross, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    lat = torch.randn(B, 4, h, h, device=DEV, generator=g)
    emb = torch.randn(2 * B, 77, cross, device=DEV, generator=g) * 0.5
    mask = (torch.rand(B, 1, h, h, device=DEV, generator=g) > 0.5).float()
    ml = torch.randn(B, 4, h, h, device=DEV, generator=g)
    ctrls = [torch.rand(B, 3, 8 * h, 8 * h, device=DEV, generator=g) for _ in range(3)]
    return lat, emb, mask, ml, ctrls


def _loops(tiny, B, h, steps, cases, seed=2, min_cos=0.998, name="tiny"):
    """cases: (n_nets, scales, keeps, guess) run through FusedDenoiser and the oracle loop on the same inputs"""
    from oracle.controlnet_multi import loop_controlnet_multi
    from powerpaint_b200.denoise import FusedDenoiser
    from powerpaint_b200.models import MultiControlNetModel

    om_u, pm_u, o = _net("unet", 9, 1234, tiny)
    cns = [_net("controlnet", 4, s, tiny) for s in (77, 78)]
    lat, emb, mask, ml, ctrls = _inputs(B, h, o.cross_attention_dim, seed)
    so, sp, ts = _scheds(steps)
    den = FusedDenoiser(pm_u, MultiControlNetModel([p for _, p, _ in cns]), "controlnet")
    for n, scales, keeps, guess in cases:
        imgs = [c if guess else torch.cat([c] * 2) for c in ctrls[:n]]
        ref = loop_controlnet_multi(om_u, [m for m, _, _ in cns[:n]], so, lat, emb, mask, ml, imgs, 7.5, scales,
                                    keeps=keeps, guess_mode=guess)
        got = den.run(latents=lat, prompt_embeds=emb, side_prompt_embeds=emb, control_image=imgs, timesteps=ts,
                      coef=sp.step_coefficients(ts), guidance_scale=7.5, extra=torch.cat([mask, ml], 1),
                      side_scale=scales, side_keep=keeps, guess_mode=guess)
        r, c = _rel(got, ref), _cos(got, ref)
        _report(f"controlnet_multi_loop_{name}", nets=n, guess=guess, rel=r, cos=c)
        assert torch.isfinite(got).all()
        assert r < 5e-2 and c > min_cos, (n, guess, r, c)
    return den


def test_loops_two_nets_and_guess_mode_tiny():
    keep2 = [[1.0] * 8, [0.0, 0.0, 1.0, 1.0, 1.0, 1.0, 0.0, 0.0]]
    _loops(True, 2, 8, 8, [(2, [0.5, 0.8], keep2, False), (1, [0.7], None, True), (2, [0.6, 0.9], keep2, True)])


def test_loops_two_nets_and_guess_mode_sd15_c5():
    """the C5 per-GPU shape: 2 images at 512x512 (64x64 latents) x CFG, 5 DDIM steps"""
    _loops(False, 2, 64, 5, [(2, [0.5, 0.8], None, False), (1, [0.5], None, True), (2, [0.5, 0.8], None, True)],
           min_cos=0.999, name="sd15_c5")


def test_residual_sum_identities_are_exact():
    """a one-net MultiControlNetModel is the single ControlNet bit for bit; a second net at scale 0 or outside its
    guidance window adds exactly zero"""
    from powerpaint_b200.denoise import FusedDenoiser
    from powerpaint_b200.models import MultiControlNetModel

    _, pm_u, o = _net("unet", 9, 1234)
    (_, a, _), (_, b, _) = _net("controlnet", 4, 77), _net("controlnet", 4, 78)
    lat, emb, mask, ml, ctrls = _inputs(2, 8, o.cross_attention_dim, 5)
    _, sp, ts = _scheds(6)
    c0, c1 = torch.cat([ctrls[0]] * 2), torch.cat([ctrls[1]] * 2)
    keep = [1.0, 1.0, 1.0, 0.0, 1.0, 1.0]
    kw = dict(latents=lat, prompt_embeds=emb, side_prompt_embeds=emb, timesteps=ts, coef=sp.step_coefficients(ts),
              guidance_scale=7.5, extra=torch.cat([mask, ml], 1))
    single = FusedDenoiser(pm_u, a, "controlnet").run(control_image=c0, side_scale=0.6, side_keep=keep, **kw)
    one = FusedDenoiser(pm_u, MultiControlNetModel([a]), "controlnet").run(control_image=[c0], side_scale=[0.6],
                                                                           side_keep=[keep], **kw)
    assert torch.equal(one, single)
    den2 = FusedDenoiser(pm_u, MultiControlNetModel([a, b]), "controlnet")
    zero_scale = den2.run(control_image=[c0, c1], side_scale=[0.6, 0.0], side_keep=[keep, None], **kw)
    assert torch.equal(zero_scale, single)
    no_window = den2.run(control_image=[c0, c1], side_scale=[0.6, 0.9], side_keep=[keep, [0.0] * 6], **kw)
    assert torch.equal(no_window, single)
    both = den2.run(control_image=[c0, c1], side_scale=[0.6, 0.9], side_keep=[keep, None], **kw)
    assert not torch.equal(both, single)


def test_controlnet_forward_guess_mode_vs_oracle():
    from oracle.controlnet_multi import controlnet_forward

    om, pm, o = _net("controlnet", 4, 77)
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(2, 4, 8, 8, device=DEV, generator=g)
    ctx = torch.randn(2, 77, o.cross_attention_dim, device=DEV, generator=g) * 0.5
    cond = torch.rand(2, 3, 64, 64, device=DEV, generator=g)
    for guess in (True, False):
        rd, rm = controlnet_forward(om, x, 321, ctx, cond, 0.8, guess)
        gd, gm = pm(x, 321, ctx, cond, conditioning_scale=0.8, guess_mode=guess, return_dict=False)
        for r, gt in zip(rd + [rm], gd + [gm]):
            assert _rel(gt, r) < 3e-2, (guess, _rel(gt, r))
    # the first down residual carries 0.1 x the scale in guess mode: the plans differ only in those constants
    assert _rel(pm(x, 321, ctx, cond, 0.8, guess_mode=True).down_block_res_samples[0],
                0.1 * pm(x, 321, ctx, cond, 0.8).down_block_res_samples[0]) < 1e-2


def test_multi_controlnet_forward_sums_the_nets():
    from oracle.controlnet_multi import controlnet_forward
    from powerpaint_b200.models import MultiControlNetModel

    (oa, a, o), (ob, b, _), (_, c, _) = (_net("controlnet", 4, s) for s in (77, 78, 79))
    g = torch.Generator(device=DEV).manual_seed(4)
    x = torch.randn(2, 4, 8, 8, device=DEV, generator=g)
    ctx = torch.randn(2, 77, o.cross_attention_dim, device=DEV, generator=g) * 0.5
    ca, cb, cc = (torch.rand(2, 3, 64, 64, device=DEV, generator=g) for _ in range(3))
    for guess in (False, True):
        da, ma = controlnet_forward(oa, x, 10, ctx, ca, 0.5, guess)
        db, mb = controlnet_forward(ob, x, 10, ctx, cb, 0.9, guess)
        # zip semantics: the third net is not run for a two-entry scale list
        gd, gm = MultiControlNetModel([a, b, c])(x, 10, ctx, [ca, cb, cc], [0.5, 0.9], guess_mode=guess)
        for r, gt in zip([p + q for p, q in zip(da, db)] + [ma + mb], gd + [gm]):
            assert _rel(gt, r) < 3e-2, (guess, _rel(gt, r))


@pytest.mark.parametrize("name", ["gpu_multi", "gpu_multi_guess"])
def test_multi_call_cuda_vs_reference_call(name):
    """the public `__call__` with two ControlNets on the GPU against the reference's own `__call__`
    (ref:pipeline_PowerPaint_ControlNet.py:1349-1770 over diffusers' MultiControlNetModel)"""
    from controlnet_multi_cases import GPU_CASES, UNET_SEED, control_argument, control_images
    from pipeline_cases import sized_inputs

    from oracle.vae import AutoencoderKLOracle
    from powerpaint_b200.engine import NetConfig
    from powerpaint_b200.models import ControlNetModel, UNet2DConditionModel, synthetic_state_dict
    from powerpaint_b200.pipelines import StableDiffusionControlNetInpaintPipeline
    from powerpaint_b200.schedulers import DDIMScheduler

    def cfg(cin):
        return NetConfig(in_channels=cin, block_out_channels=(32, 64, 128, 128), attention_head_dim=4,
                         cross_attention_dim=64, norm_num_groups=8)

    def model(cls, cin, kind, seed):
        return cls.from_state_dict(cfg(cin), synthetic_state_dict(cfg(cin), kind, seed)).to(DEV)

    case = GPU_CASES[name]
    pipe = StableDiffusionControlNetInpaintPipeline(
        vae=AutoencoderKLOracle.synthetic(tiny=True).to(DEV), text_encoder=None, tokenizer=None,
        unet=model(UNet2DConditionModel, 9, "unet", UNET_SEED),
        controlnet=[model(ControlNetModel, 4, "controlnet", s) for s in case["nets"]], scheduler=DDIMScheduler(),
        safety_checker=None)
    s = case["size"]
    img, mask, pe, ne, ctl = sized_inputs(2, s, s, 64, case["seed"])
    out = pipe(image=img, mask=mask, control_image=control_argument(case["nets"], control_images(3, 2, s, s, ctl)),
               prompt_embeds=pe, negative_prompt_embeds=ne, height=s, width=s,
               generator=torch.Generator().manual_seed(case["gen_seed"]), output_type="latent", return_dict=False,
               **case["kw"])[0]
    ref = torch.from_numpy(np.load(os.path.join(HERE, "golden", "pipeline_controlnet_multi_call.npz"))
                           [f"{name}_latents"]).to(out.device)
    assert out.shape == ref.shape and torch.isfinite(out).all()
    r, c = _rel(out, ref), _cos(out, ref)
    _report(f"controlnet_multi __call__ {name}", rel=r, cos=c)
    assert r < 5e-2 and c > 0.998, (name, r, c)


def test_plan_cache_rerecords_per_net_count_and_guess_flag():
    from powerpaint_b200.denoise import FusedDenoiser
    from powerpaint_b200.models import MultiControlNetModel

    _, pm_u, o = _net("unet", 9, 1234)
    (_, a, _), (_, b, _) = _net("controlnet", 4, 77), _net("controlnet", 4, 78)
    lat, emb, mask, ml, ctrls = _inputs(1, 8, o.cross_attention_dim, 6)
    _, sp, ts = _scheds(3)
    multi = MultiControlNetModel([a, b])
    den = FusedDenoiser(pm_u, multi, "controlnet")
    den.MAX_PLANS = 8
    kw = dict(latents=lat, prompt_embeds=emb, side_prompt_embeds=emb, timesteps=ts, coef=sp.step_coefficients(ts),
              guidance_scale=7.5, extra=torch.cat([mask, ml], 1))
    c2 = [torch.cat([c] * 2) for c in ctrls[:2]]
    r1 = den.run(control_image=c2[:1], side_scale=[0.5], **kw)
    den.run(control_image=c2, side_scale=[0.5, 0.5], **kw)
    den.run(control_image=ctrls[:2], side_scale=[0.5, 0.5], guess_mode=True, **kw)
    assert len(den._cache) == 3
    assert torch.equal(den.run(control_image=c2[:1], side_scale=[0.5], **kw), r1)  # cached plan replayed
    assert len(den._cache) == 3
    b.load_state_dict(b.state_dict())  # net 1 changed: the next recording drops every plan that recorded it
    den.run(control_image=c2, side_scale=[0.5, 0.5], **kw)
    gens = ((a.generation,), (a.generation, b.generation))
    assert len(den._cache) == 2 and all(k[-1] in gens for k in den._cache)
    assert torch.equal(den.run(control_image=c2[:1], side_scale=[0.5], **kw), r1)  # the one-net plan stayed valid
    assert len(den._cache) == 2
