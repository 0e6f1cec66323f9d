"""Generate tests/golden/pipeline_v1_call.npz by running the REFERENCE's own v1 pipeline `__call__`.

    PP_REFERENCE_DIR=<checkout of the original PowerPaint project> python tests/golden/make_pipeline_golden.py

`powerpaint/pipelines/pipeline_PowerPaint.py` of that checkout and the reference UNet are imported UNMODIFIED over
tests/golden/diffusers_shim. What the fixture pins is everything `__call__` itself does between the user's arguments and
the final latents (pipeline_PowerPaint.py:855-1071): `prepare_mask_and_masked_image`, the strength -> timestep window,
the order of the generator draws (initial noise first, then the VAE posterior sample of the masked image), the mask
interpolation, the CFG duplication, `cat([latents, mask, masked_image_latents])`, the guidance formula, the scheduler
call contract. The VAE and the DDIM scheduler behind the diffusers names are the oracle's (oracle/vae.py,
oracle/ddim.py), the UNet is the reference's with the synthetic weights; prompts enter as embeddings so no tokenizer
or text encoder is involved (`_encode_prompt` :317-470 only concatenates them, negative first).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(HERE, "diffusers_shim"), os.environ["PP_REFERENCE_DIR"], ROOT]

import types  # noqa: E402

_mm = types.ModuleType("mmengine")  # powerpaint/utils/utils.py:12 imports mmengine.print_log (absent here)
_mm.print_log = lambda *a, **k: None
sys.modules.setdefault("mmengine", _mm)

from diffusers.models import AutoencoderKL  # noqa: E402  (shim: the oracle VAE)
from diffusers.schedulers import DDIMScheduler  # noqa: E402  (shim: the oracle DDIM)
from powerpaint.models.unet_2d_condition import UNet2DConditionModel as RefUNet  # noqa: E402  (reference, unmodified)
from powerpaint.pipelines.pipeline_PowerPaint import StableDiffusionInpaintPipeline as RefPipe  # noqa: E402
from powerpaint.pipelines.pipeline_PowerPaint import prepare_mask_and_masked_image as ref_prepare  # noqa: E402

from make_unet_golden import CROSS, cfg, ref_unet  # noqa: E402
from powerpaint_b200.models import synthetic_state_dict  # noqa: E402

CASES = {  # name -> (strength, steps, guidance, eta, per-sample generators)
    "full": (1.0, 4, 7.5, 0.0, False),
    "strength_half": (0.5, 8, 7.5, 0.0, False),
    "no_cfg_genlist": (1.0, 3, 1.0, 0.0, True),
    "eta_half": (1.0, 3, 7.5, 0.5, False),  # the scheduler draws its variance noise from the same generator
}
B, H, W = 2, 64, 48


def call_inputs():
    g = torch.Generator().manual_seed(9)
    img = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    mask = torch.zeros(B, 1, H, W)
    mask[0, :, 8:40, 16:40] = 1
    mask[1, :, 20:60, 4:30] = 0.7  # binarised at 0.5 by prepare_mask_and_masked_image
    pe = torch.randn(B, 77, CROSS, generator=g) * 0.5
    ne = torch.randn(B, 77, CROSS, generator=g) * 0.5
    return img, mask, pe, ne


PROMPTS = dict(promptA=["a photo of a cat P_obj", "the dog on the wall"], promptB=["a photo of a cat", "empty scene blur"],
               promptU=["a chair on the wall", "sky"], negative_promptA=["blur", "a dog"],
               negative_promptB=["empty scene", "a dog"], negative_promptU=["blur wall", ""])


def text_stack():
    """one synthetic tokenizer, two synthetic CLIP text encoders of the UNet's cross-attention width"""
    from synthetic_clip import make_text_encoder, make_tokenizer

    tok = make_tokenizer()
    return tok, make_text_encoder(len(tok), hidden=CROSS, seed=1), make_text_encoder(len(tok), hidden=CROSS, seed=2)


def brushnet_inputs():
    """image in [0, 1] (normalised by prepare_image), mask in [0, 1] whose ZEROS mark the hole (-1 after normalising,
    `sum(1) < 0` :1308)"""
    g = torch.Generator().manual_seed(21)
    img = torch.rand(B, 3, H, W, generator=g)
    mask = torch.ones(B, 3, H, W)
    mask[0, :, 8:40, 16:40] = 0
    mask[1, :, 20:60, 4:30] = 0
    return img * mask, mask


def generators(per_sample):
    return [torch.Generator().manual_seed(40 + i) for i in range(B)] if per_sample else torch.Generator().manual_seed(4)


@torch.no_grad()
def main():
    unet = ref_unet(9)
    unet.load_state_dict(synthetic_state_dict(cfg(9), "unet", 77), strict=True)
    pipe = RefPipe(vae=AutoencoderKL.synthetic(tiny=True), text_encoder=None, tokenizer=None, unet=unet,
                   scheduler=DDIMScheduler(), safety_checker=None, feature_extractor=None, requires_safety_checker=False)
    img, mask, pe, ne = call_inputs()
    out = {}
    m, mi, init = ref_prepare(img, mask, H, W, return_image=True)
    out["prepare_mask"], out["prepare_masked_image"], out["prepare_image"] = m.numpy(), mi.numpy(), init.numpy()
    # the same through the numpy / PIL entry of prepare_mask_and_masked_image (uint8 HWC image, HW mask in [0,1])
    rng = np.random.default_rng(5)
    img_u8 = rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8)
    mask_np = (rng.random((H, W)) > 0.6).astype(np.float32)
    m2, mi2 = ref_prepare(img_u8, mask_np, H, W)
    out["prepare_np_mask"], out["prepare_np_masked_image"] = m2.numpy(), mi2.numpy()
    # every input container prepare_mask_and_masked_image accepts, as digests (bit-exact without storing the tensors)
    import json

    from pipeline_cases import digest_prepare, prepare_input_kinds

    kinds = {k: digest_prepare(ref_prepare, i, m, H, W) for k, (i, m) in prepare_input_kinds(H, W).items()}
    with open(os.path.join(os.environ.get("PP_GOLDEN_OUT", HERE), "prepare_input_kinds.json"), "w") as f:
        json.dump(kinds, f, indent=1, sort_keys=True)
    for name, (strength, steps, gs, eta, per_sample) in CASES.items():
        seen = []
        lat = pipe(image=img, mask=mask, prompt_embeds=pe, negative_prompt_embeds=ne, height=H, width=W,
                   strength=strength, num_inference_steps=steps, guidance_scale=gs, eta=eta,
                   generator=generators(per_sample), output_type="latent", return_dict=False,
                   callback=lambda i, t, x: seen.append(int(t)))[0]
        out[f"{name}_latents"] = lat.numpy()
        out[f"{name}_timesteps"] = np.array(seen, dtype=np.int64)
        print(name, tuple(lat.shape), seen, float(lat.abs().mean()))
    # two images per prompt (prompts repeat interleaved :441-443, masks / masked images tile :685-698) from caller latents
    lat0 = torch.randn(2 * B, 4, H // 8, W // 8, generator=torch.Generator().manual_seed(77))
    lat = pipe(image=img, mask=mask, prompt_embeds=pe, negative_prompt_embeds=ne, height=H, width=W,
               num_images_per_prompt=2, latents=lat0, num_inference_steps=2, guidance_scale=7.5,
               generator=generators(False), output_type="latent", return_dict=False)[0]
    out["per_prompt2_latents"] = lat.numpy()
    # fixtures for the GPU tests (tests/test_golden_gpu.py): same call, latent sizes the tiny GPU tests already exercise
    from pipeline_cases import GPU_V1, GPU_V1_STRENGTH, sized_inputs

    for name, case in (("gpu_v1", GPU_V1), ("gpu_v1_strength", GPU_V1_STRENGTH)):
        gi, gm, gpe, gne, _ = sized_inputs(B, case["size"], case["size"], CROSS, case["seed"])
        lat = pipe(image=gi, mask=gm, prompt_embeds=gpe, negative_prompt_embeds=gne, height=case["size"],
                   width=case["size"], generator=torch.Generator().manual_seed(case["gen_seed"]), output_type="latent",
                   return_dict=False, **case["kw"])[0]
        out[f"{name}_latents"] = lat.numpy()
        print(name, tuple(lat.shape), float(lat.abs().mean()))
    # what the reference raises for invalid calls (check_inputs :554-602, prepare_mask_and_masked_image :39-153, ...)
    from pipeline_cases import error_cases

    record_errors(pipe, error_cases(img, mask, pe, ne, H, W), "pipeline_v1_errors.json")
    # string prompts through the reference's `_encode_prompt` (tokenizer + text encoder, A/B trade-off :317-470)
    tok, te, _ = text_stack()
    pipe_t = RefPipe(vae=AutoencoderKL.synthetic(tiny=True), text_encoder=te, tokenizer=tok, unet=unet,
                     scheduler=DDIMScheduler(), safety_checker=None, feature_extractor=None,
                     requires_safety_checker=False)
    lat = pipe_t(promptA=PROMPTS["promptA"], promptB=PROMPTS["promptB"], tradoff=0.7, tradoff_nag=0.4,
                 negative_promptA=PROMPTS["negative_promptA"], negative_promptB=PROMPTS["negative_promptB"], image=img,
                 mask=mask, height=H, width=W, num_inference_steps=3, guidance_scale=7.5,
                 generator=generators(False), output_type="latent", return_dict=False)[0]
    out["prompts_latents"] = lat.numpy()
    # 4-channel UNet: no mask channels; after every step the known region is reset to the noised original (:1025-1035,
    # which indexes image_latents[:1] and mask[:1] — sample 0's image and mask serve the whole batch)
    u4 = ref_unet(4)
    u4.load_state_dict(synthetic_state_dict(cfg(4), "unet", 78), strict=True)
    pipe4 = RefPipe(vae=AutoencoderKL.synthetic(tiny=True), text_encoder=None, tokenizer=None, unet=u4,
                    scheduler=DDIMScheduler(), safety_checker=None, feature_extractor=None,
                    requires_safety_checker=False)
    for name, strength, steps in (("unet4_full", 1.0, 3), ("unet4_strength", 0.6, 5)):
        lat = pipe4(image=img, mask=mask, prompt_embeds=pe, negative_prompt_embeds=ne, height=H, width=W,
                    strength=strength, num_inference_steps=steps, guidance_scale=7.5, generator=generators(False),
                    output_type="latent", return_dict=False)[0]
        out[f"{name}_latents"] = lat.numpy()
        print(name, tuple(lat.shape), float(lat.abs().mean()))
    save("pipeline_v1_call.npz", out)
    brushnet_golden()
    controlnet_golden()


def record_errors(pipe, cases, name):
    import json

    errors = {}
    for case, kw in cases.items():
        try:
            pipe(**kw)
            errors[case] = ["no error", ""]
        except Exception as e:  # noqa: BLE001  (recording whatever the reference raises is the point)
            errors[case] = [type(e).__name__, str(e)]
    with open(os.path.join(os.environ.get("PP_GOLDEN_OUT", HERE), name), "w") as f:
        json.dump(errors, f, indent=1, sort_keys=True)
    print("wrote", name, sum(v[0] != "no error" for v in errors.values()), "errors of", len(errors), "cases")


def save(name, out):
    path = os.path.join(os.environ.get("PP_GOLDEN_OUT", HERE), name)  # (the staleness test writes elsewhere)
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


@torch.no_grad()
def brushnet_golden():
    """v2: the reference's `StableDiffusionPowerPaintBrushNetPipeline.__call__` (pipeline_PowerPaint_Brushnet_CA.py:
    1026-1497) with the reference's UNet AND BrushNet; promptU always goes through tokenizer + text encoder (:1262)"""
    import copy

    from powerpaint.models.BrushNet_CA import BrushNetModel as RefBrushNet
    from powerpaint.pipelines.pipeline_PowerPaint_Brushnet_CA import StableDiffusionPowerPaintBrushNetPipeline as RefBN

    u4 = ref_unet(4)
    u4.load_state_dict(synthetic_state_dict(cfg(4), "unet", 11), strict=True)
    bn = copy.deepcopy(RefBrushNet.from_unet(ref_unet(4), conditioning_channels=5)).eval()
    bn.load_state_dict(synthetic_state_dict(cfg(4), "brushnet", 12), strict=True)
    tok, te, te_b = text_stack()
    pipe = RefBN(vae=AutoencoderKL.synthetic(tiny=True), text_encoder=te, text_encoder_brushnet=te_b, tokenizer=tok,
                 unet=u4, brushnet=bn, scheduler=DDIMScheduler(), safety_checker=None, feature_extractor=None,
                 requires_safety_checker=False)
    img, mask = brushnet_inputs()
    out = {}
    for name, kw in BRUSHNET_CASES.items():
        torch.manual_seed(123)  # the conditioning latents are sampled from the GLOBAL generator (:1335)
        lat = pipe(**PROMPTS, tradoff=0.7, tradoff_nag=0.4, image=img, mask=mask, generator=generators(False),
                   output_type="latent", return_dict=False, **kw)[0]
        out[f"{name}_latents"] = lat.numpy()
        print("brushnet", name, tuple(lat.shape), float(lat.abs().mean()))
    save("pipeline_brushnet_call.npz", out)
    from pipeline_cases import brushnet_error_cases

    record_errors(pipe, brushnet_error_cases(img, mask, PROMPTS, CROSS), "pipeline_brushnet_errors.json")


BRUSHNET_CASES = {
    "full": dict(num_inference_steps=3, guidance_scale=7.5, brushnet_conditioning_scale=1.0),
    "window_scale": dict(num_inference_steps=4, guidance_scale=5.0, brushnet_conditioning_scale=0.8,
                         control_guidance_start=0.0, control_guidance_end=0.6),
    "per_prompt2": dict(num_inference_steps=2, guidance_scale=7.5, brushnet_conditioning_scale=1.0,
                        num_images_per_prompt=2),
    # (guidance_scale <= 1 is not a case: the reference's encode_prompt concatenates a None then, :627)
}
CONTROLNET_CASES = {
    "full": dict(strength=1.0, num_inference_steps=3, guidance_scale=5.0, controlnet_conditioning_scale=0.5),
    "strength_window": dict(strength=0.5, num_inference_steps=6, guidance_scale=7.5, controlnet_conditioning_scale=0.8,
                            control_guidance_start=0.3, control_guidance_end=1.0),
    "per_prompt2": dict(strength=1.0, num_inference_steps=2, guidance_scale=7.5, controlnet_conditioning_scale=0.5,
                        num_images_per_prompt=2),
}


@torch.no_grad()
def controlnet_golden():
    """ControlNet: the reference's `StableDiffusionControlNetInpaintPipeline.__call__`
    (pipeline_PowerPaint_ControlNet.py:1349-1770) with the reference's UNet; the ControlNet behind the diffusers name
    is the oracle's (it lives in diffusers, not in the reference)"""
    from diffusers.models import ControlNetModel
    from oracle.unet import UNetConfig
    from powerpaint.pipelines.pipeline_PowerPaint_ControlNet import StableDiffusionControlNetInpaintPipeline as RefCN

    u9 = ref_unet(9)
    u9.load_state_dict(synthetic_state_dict(cfg(9), "unet", 5), strict=True)
    cn = ControlNetModel(UNetConfig.tiny(4)).eval()
    cn.load_state_dict(synthetic_state_dict(cfg(4), "controlnet", 6), strict=True)
    pipe = RefCN(vae=AutoencoderKL.synthetic(tiny=True), text_encoder=None, tokenizer=None, unet=u9, controlnet=cn,
                 scheduler=DDIMScheduler(), safety_checker=None, feature_extractor=None, requires_safety_checker=False)
    img, mask, pe, ne = call_inputs()
    ctl = torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(31))
    out = {}
    for name, kw in CONTROLNET_CASES.items():
        lat = pipe(image=img, mask=mask, control_image=ctl, prompt_embeds=pe, negative_prompt_embeds=ne, height=H,
                   width=W, generator=generators(False), output_type="latent", return_dict=False, **kw)[0]
        out[f"{name}_latents"] = lat.numpy()
        print("controlnet", name, tuple(lat.shape), float(lat.abs().mean()))
    from pipeline_cases import GPU_CONTROLNET as case, sized_inputs

    gi, gm, gpe, gne, gctl = sized_inputs(B, case["size"], case["size"], CROSS, case["seed"])
    lat = pipe(image=gi, mask=gm, control_image=gctl, prompt_embeds=gpe, negative_prompt_embeds=gne,
               height=case["size"], width=case["size"], generator=torch.Generator().manual_seed(case["gen_seed"]),
               output_type="latent", return_dict=False, **case["kw"])[0]
    out["gpu_controlnet_latents"] = lat.numpy()
    print("gpu_controlnet", tuple(lat.shape), float(lat.abs().mean()))
    save("pipeline_controlnet_call.npz", out)
    from pipeline_cases import controlnet_error_cases

    img, mask, pe, ne = call_inputs()
    record_errors(pipe, controlnet_error_cases(img, mask, pe, ne, ctl, H, W), "pipeline_controlnet_errors.json")


if __name__ == "__main__":
    main()
