"""CPU tests of several ControlNets and ControlNet guess mode: the product's `__call__` host side against the final
latents of the reference's own `__call__` (tests/golden/pipeline_controlnet_multi_call.npz, generator
tests/golden/make_controlnet_multi_golden.py), its invalid calls against what the reference raises, the
MultiControlNetModel checkpoint layout, and `sharded_call` with one control image per ControlNet.

The fused denoiser is replaced by `_MultiControlNetCoefficientDenoiser`, an fp32 stand-in over the oracle nets that
takes the keywords the pipeline hands `FusedDenoiser.run` (lists per net, `guess_mode`), so a difference can only come
from the pipeline's host code or the stand-in."""
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))

from controlnet_multi_cases import (CASES, GPU_CASES, UNET_SEED, control_argument, control_images,  # noqa: E402
                                    error_cases)

BOC, HEADS, CROSS, GROUPS = (32, 64, 128, 128), 4, 64, 8
B, H, W = 2, 64, 48


def _cfg(cin):
    from powerpaint_b200.engine import NetConfig

    return NetConfig(in_channels=cin, block_out_channels=BOC, attention_head_dim=HEADS, cross_attention_dim=CROSS,
                     norm_num_groups=GROUPS)


def _oracle(cls, cin, kind, seed):
    from oracle.unet import UNetConfig
    from powerpaint_b200.models import synthetic_state_dict

    sd = synthetic_state_dict(_cfg(cin), kind, seed)
    m = cls(UNetConfig.tiny(cin)).eval()
    m.load_state_dict(sd, strict=True)
    return m, sd


def _rel(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12))


class _MultiControlNetCoefficientDenoiser:
    """stand-in for FusedDenoiser(mode="controlnet").run with one or several ControlNets and guess mode: oracle nets,
    coefficient-row DDIM"""

    def __init__(self, unet, controlnets):
        self.unet, self.controlnets = unet, controlnets
        self.calls = []

    @torch.no_grad()
    def run(self, *, latents, prompt_embeds, side_prompt_embeds, control_image, timesteps, coef, guidance_scale,
            extra, side_scale, side_keep=None, noise_fn=None, callback=None, ucoef=None, guess_mode=False):
        from oracle.controlnet_multi import controlnet_forward

        self.calls.append(dict(multi=isinstance(control_image, list), guess_mode=guess_mode))
        multi = isinstance(control_image, list)
        images = control_image if multi else [control_image]
        scales = side_scale if multi else [side_scale]
        keeps = side_keep if multi else [side_keep]
        do_cfg = guidance_scale > 1.0
        half = guess_mode and do_cfg
        for i, t in enumerate(timesteps):
            x4 = torch.cat([latents] * 2) if do_cfg else latents
            ex = torch.cat([extra] * 2) if do_cfg else extra
            xc, pc = (latents, side_prompt_embeds[latents.shape[0]:]) if half else (x4, side_prompt_embeds)
            d = m = None
            for net, img, s, kp in zip(self.controlnets, images, scales, keeps):
                scale = s * (kp[i] if kp is not None else 1.0)
                dk, mk = controlnet_forward(net, xc, int(t), pc, img, scale, guess_mode)
                d, m = (dk, mk) if d is None else ([a + b for a, b in zip(d, dk)], m + mk)
            if half:
                d = [torch.cat([torch.zeros_like(r), r]) for r in d]
                m = torch.cat([torch.zeros_like(m), m])
            eps = self.unet(torch.cat([x4, ex], dim=1), int(t), prompt_embeds, down_block_additional_residuals=d,
                            mid_block_additional_residual=m)
            if do_cfg:
                u, c = eps.chunk(2)
                eps = u + guidance_scale * (c - u)
            sa, s1a, sap, dirc, _ = [float(v) for v in coef[i, :5]]
            latents = sap * ((latents - s1a * eps) / sa) + dirc * eps
        return latents


def _pipe(nets):
    """product pipeline over the case's ControlNets (tuple of weight seeds -> a list, int -> one net), stand-in loop"""
    from oracle.unet import ControlNetOracle, UNet2DConditionOracle
    from oracle.vae import AutoencoderKLOracle
    from powerpaint_b200.models import ControlNetModel, UNet2DConditionModel
    from powerpaint_b200.pipelines import StableDiffusionControlNetInpaintPipeline
    from powerpaint_b200.schedulers import DDIMScheduler

    ou, sd_u = _oracle(UNet2DConditionOracle, 9, "unet", UNET_SEED)
    seeds = nets if isinstance(nets, tuple) else (nets,)
    oracles = [_oracle(ControlNetOracle, 4, "controlnet", s) for s in seeds]
    prod = [ControlNetModel.from_state_dict(_cfg(4), sd) for _, sd in oracles]
    pipe = StableDiffusionControlNetInpaintPipeline(
        vae=AutoencoderKLOracle.synthetic(tiny=True), text_encoder=None, tokenizer=None,
        unet=UNet2DConditionModel.from_state_dict(_cfg(9), sd_u),
        controlnet=prod if isinstance(nets, tuple) else prod[0], scheduler=DDIMScheduler())
    fake = _MultiControlNetCoefficientDenoiser(ou, [o for o, _ in oracles])
    pipe.denoiser = lambda: fake
    return pipe, fake


def _call_inputs():  # == make_pipeline_golden.call_inputs
    g = torch.Generator().manual_seed(9)
    img = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    mask = torch.zeros(B, 1, H, W)
    mask[0, :, 8:40, 16:40] = 1
    mask[1, :, 20:60, 4:30] = 0.7
    pe = torch.randn(B, 77, CROSS, generator=g) * 0.5
    ne = torch.randn(B, 77, CROSS, generator=g) * 0.5
    return img, mask, pe, ne


@pytest.mark.parametrize("name", sorted(CASES))
def test_multi_and_guess_call_equals_reference_call_golden(name):
    gold = np.load(os.path.join(HERE, "golden", "pipeline_controlnet_multi_call.npz"))
    case = CASES[name]
    pipe, fake = _pipe(case["nets"])
    img, mask, pe, ne = _call_inputs()
    ctls = control_images(3, B, H, W)
    out = pipe(image=img, mask=mask, control_image=control_argument(case["nets"], ctls), prompt_embeds=pe,
               negative_prompt_embeds=ne, height=H, width=W, generator=torch.Generator().manual_seed(4),
               output_type="latent", return_dict=False, **case["kw"])[0]
    ref = torch.from_numpy(gold[f"{name}_latents"])
    assert out.shape == ref.shape and _rel(out, ref) < 5e-5, _rel(out, ref)
    assert fake.calls[-1]["guess_mode"] == case["kw"].get("guess_mode", False)


@pytest.mark.parametrize("name", sorted(GPU_CASES))
def test_gpu_multi_fixture_cases_on_the_cpu_stand_in(name):
    """the fixtures tests/test_controlnet_multi_gpu.py holds the CUDA path to, first through the fp32 stand-in"""
    from pipeline_cases import sized_inputs

    gold = np.load(os.path.join(HERE, "golden", "pipeline_controlnet_multi_call.npz"))
    case = GPU_CASES[name]
    pipe, _ = _pipe(case["nets"])
    s = case["size"]
    img, mask, pe, ne, ctl = sized_inputs(B, s, s, CROSS, case["seed"])
    out = pipe(image=img, mask=mask, control_image=control_argument(case["nets"], control_images(3, B, s, s, ctl)),
               prompt_embeds=pe, negative_prompt_embeds=ne, height=s, width=s,
               generator=torch.Generator().manual_seed(case["gen_seed"]), output_type="latent", return_dict=False,
               **case["kw"])[0]
    assert _rel(out, torch.from_numpy(gold[f"{name}_latents"])) < 5e-5


def test_multi_controlnet_invalid_calls_raise_what_the_reference_raises():
    with open(os.path.join(HERE, "golden", "pipeline_controlnet_multi_errors.json")) as f:
        gold = json.load(f)
    pipe, _ = _pipe((6, 7))
    img, mask, pe, ne = _call_inputs()
    cases = error_cases(img, mask, pe, ne, control_images(3, B, H, W), H, W)
    assert sorted(cases) == sorted(gold) and all(v[0] != "no error" for v in gold.values())
    for name, kw in cases.items():
        kind, msg = gold[name]
        with pytest.raises(Exception) as ei:
            pipe(**kw)
        assert (type(ei.value).__name__, str(ei.value)) == (kind, msg), name


def test_single_controlnet_passes_the_keywords_it_always_did():
    """one ControlNetModel without guess mode: `run` gets no list and no `guess_mode` keyword"""
    pipe, fake = _pipe(6)
    img, mask, pe, ne = _call_inputs()
    seen = {}
    orig = fake.run

    def spy(**kw):
        seen.update(kw)
        return orig(**kw)
    fake.run = spy
    pipe(image=img, mask=mask, control_image=control_images(1, B, H, W)[0], prompt_embeds=pe, negative_prompt_embeds=ne,
         height=H, width=W, num_inference_steps=2, controlnet_conditioning_scale=0.5, output_type="latent")
    assert sorted(seen) == sorted(["latents", "prompt_embeds", "side_prompt_embeds", "control_image", "timesteps",
                                   "coef",
                                   "guidance_scale", "extra", "side_scale", "side_keep", "noise_fn", "ucoef",
                                   "callback"])
    assert isinstance(seen["side_scale"], float) and torch.is_tensor(seen["control_image"])


@pytest.mark.parametrize("container", [list, tuple])
def test_pipeline_wraps_a_list_or_tuple_of_controlnets(container):
    from powerpaint_b200.models import ControlNetModel, MultiControlNetModel, UNet2DConditionModel
    from powerpaint_b200.pipelines import StableDiffusionControlNetInpaintPipeline
    from powerpaint_b200.schedulers import DDIMScheduler

    nets = [ControlNetModel(_cfg(4)) for _ in range(2 if container is list else 1)]
    pipe = StableDiffusionControlNetInpaintPipeline(vae=None, text_encoder=None, tokenizer=None,
                                                    unet=UNet2DConditionModel(_cfg(9)), controlnet=container(nets),
                                                    scheduler=DDIMScheduler())
    assert isinstance(pipe.controlnet, MultiControlNetModel)
    assert list(pipe.controlnet.nets) == nets
    assert pipe.controlnet.config.global_pool_conditions is False


def test_multi_controlnet_generation_follows_every_net():
    from powerpaint_b200.models import ControlNetModel, MultiControlNetModel

    a, b = ControlNetModel(_cfg(4)), ControlNetModel(_cfg(4))
    m = MultiControlNetModel([a, b])
    g0 = m.generation
    b.load_state_dict(b.state_dict())
    assert m.generation != g0
    g1 = m.generation
    m.to(torch.float16)  # output dtype only: parameters untouched
    assert m.dtype == torch.float16 and a.dtype == torch.float16 and m.generation == g1


def test_multi_controlnet_save_load_round_trip(tmp_path):
    from powerpaint_b200.models import ControlNetModel, MultiControlNetModel, synthetic_state_dict

    nets = [ControlNetModel.from_state_dict(_cfg(4), synthetic_state_dict(_cfg(4), "controlnet", s)) for s in (6, 7, 8)]
    d = str(tmp_path / "cn")
    MultiControlNetModel(nets).save_pretrained(d)
    assert sorted(os.listdir(tmp_path)) == ["cn", "cn_1", "cn_2"]
    back = MultiControlNetModel.from_pretrained(d)
    assert len(back.nets) == 3
    for n0, n1 in zip(nets, back.nets):
        sd0, sd1 = n0.state_dict(), n1.state_dict()
        assert sorted(sd0) == sorted(sd1) and all(torch.equal(sd0[k], sd1[k]) for k in sd0)
    one = MultiControlNetModel.from_pretrained(str(tmp_path / "cn_2"))  # no cn_2_1 next to it
    assert len(one.nets) == 1
    with pytest.raises(ValueError, match="No ControlNets found"):
        MultiControlNetModel.from_pretrained(str(tmp_path / "missing"))


# ---------------------------------------------------------------- sharded_call with a list of control images
def _sharded_worker(rank, world, port, q):
    import torch.distributed as dist

    from powerpaint_b200.parallel import sharded_call

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        pipe, _ = _pipe((6, 7))
        img, mask, pe, ne = _call_inputs()
        ctls = control_images(2, B, H, W)
        common = dict(height=H, width=W, num_inference_steps=2, guidance_scale=7.5,
                      controlnet_conditioning_scale=[0.5, 0.8], output_type="latent")
        batched = dict(image=img, mask=mask, prompt_embeds=pe, negative_prompt_embeds=ne, control_image=ctls)
        out = sharded_call(pipe, batched if rank == 0 else None, "cpu", seeds=[40, 41], **common)
        if rank == 0:
            ref = torch.cat([pipe(image=img[i:i + 1], mask=mask[i:i + 1], prompt_embeds=pe[i:i + 1],
                                  negative_prompt_embeds=ne[i:i + 1], control_image=[c[i:i + 1] for c in ctls],
                                  generator=[torch.Generator().manual_seed(40 + i)], return_dict=False, **common)[0]
                             for i in range(B)])
            q.put(("ok", _rel(out, ref), tuple(out.shape)))
    except Exception as e:  # noqa: BLE001  (reported to the parent process)
        q.put(("error", repr(e), None))
        raise
    finally:
        dist.destroy_process_group()


def test_sharded_call_scatters_a_list_of_control_images_over_gloo():
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    status, rel, shape = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
    assert status == "ok", rel
    assert shape == (B, 4, H // 8, W // 8) and rel < 1e-6, rel


def test_split_batched_lists_round_trip():
    from powerpaint_b200.parallel import _merge_shards, _split_batched

    a, b, c = torch.randn(3, 2), torch.randn(3, 4), torch.randn(3, 1)
    names, halves, tensors = _split_batched({"x": a, "control_image": [b, c]}, 3)
    kw = _merge_shards(names, halves, tensors)
    assert torch.equal(kw["x"], a) and isinstance(kw["control_image"], list)
    assert [t.shape for t in kw["control_image"]] == [b.shape, c.shape]
    with pytest.raises(ValueError):
        _split_batched({"control_image": [b, torch.randn(2, 4)]}, 3)
