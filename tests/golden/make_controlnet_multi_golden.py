"""Generate tests/golden/pipeline_controlnet_multi_call.npz and pipeline_controlnet_multi_errors.json by running the
REFERENCE's own ControlNet pipeline `__call__` with several ControlNets and with guess mode.

    PP_REFERENCE_DIR=<checkout of the original PowerPaint project> python tests/golden/make_controlnet_multi_golden.py

Same set-up as `controlnet_golden` in make_pipeline_golden.py (the reference's pipeline file and UNet unmodified over
tests/golden/diffusers_shim, the oracle ControlNet behind diffusers' name), plus diffusers_multi_controlnet.py: the
ControlNet gains diffusers' guess-mode scales, and the list of ControlNets is wrapped by the reference constructor in
diffusers' `MultiControlNetModel` (0.27: zip of images, scales and nets, residuals summed in net order). Cases:
tests/golden/controlnet_multi_cases.py. Writes pipeline_controlnet_multi_call.npz and
pipeline_controlnet_multi_errors.json only (to `$PP_GOLDEN_OUT` when set).
"""
import os
import sys

import numpy as np
import torch

import make_pipeline_golden as mpg  # noqa: E402  (puts the shim, the reference and the repository on sys.path)


@torch.no_grad()
def main():
    import diffusers_multi_controlnet
    from controlnet_multi_cases import CASES, GPU_CASES, UNET_SEED, control_argument, control_images, error_cases
    from diffusers.models import AutoencoderKL
    from diffusers_multi_controlnet import ControlNetModel

    diffusers_multi_controlnet.install()
    from diffusers.schedulers import DDIMScheduler
    from oracle.unet import UNetConfig
    from pipeline_cases import sized_inputs
    from powerpaint.pipelines.pipeline_PowerPaint_ControlNet import StableDiffusionControlNetInpaintPipeline as RefCN

    from powerpaint_b200.models import synthetic_state_dict

    u9 = mpg.ref_unet(9)
    u9.load_state_dict(synthetic_state_dict(mpg.cfg(9), "unet", UNET_SEED), strict=True)

    def net(seed):
        cn = ControlNetModel(UNetConfig.tiny(4)).eval()
        cn.load_state_dict(synthetic_state_dict(mpg.cfg(4), "controlnet", seed), strict=True)
        return cn

    def pipe(nets):
        cn = [net(s) for s in nets] if isinstance(nets, tuple) else net(nets)
        return RefCN(vae=AutoencoderKL.synthetic(tiny=True), text_encoder=None, tokenizer=None, unet=u9, controlnet=cn,
                     scheduler=DDIMScheduler(), safety_checker=None, feature_extractor=None,
                     requires_safety_checker=False)

    B, H, W = mpg.B, mpg.H, mpg.W
    img, mask, pe, ne = mpg.call_inputs()
    ctls = control_images(3, B, H, W)
    out, errors = {}, {}
    for name, case in CASES.items():
        try:
            lat = pipe(case["nets"])(image=img, mask=mask, control_image=control_argument(case["nets"], ctls),
                                     prompt_embeds=pe, negative_prompt_embeds=ne, height=H, width=W,
                                     generator=mpg.generators(False), output_type="latent", return_dict=False,
                                     **case["kw"])[0]
        except Exception as e:  # noqa: BLE001  (a call the reference cannot run is recorded as its error)
            errors[name] = [type(e).__name__, str(e)]
            print("controlnet multi", name, "raises", errors[name])
            continue
        out[f"{name}_latents"] = lat.numpy()
        print("controlnet multi", name, tuple(lat.shape), float(lat.abs().mean()))
    for name, case in GPU_CASES.items():
        s = case["size"]
        gi, gm, gpe, gne, gctl = sized_inputs(B, s, s, mpg.CROSS, case["seed"])
        lat = pipe(case["nets"])(image=gi, mask=gm, control_image=control_argument(case["nets"],
                                                                                   control_images(3, B, s, s, gctl)),
                                 prompt_embeds=gpe, negative_prompt_embeds=gne, height=s, width=s,
                                 generator=torch.Generator().manual_seed(case["gen_seed"]), output_type="latent",
                                 return_dict=False, **case["kw"])[0]
        out[f"{name}_latents"] = lat.numpy()
        print("controlnet multi", name, tuple(lat.shape), float(lat.abs().mean()))
    mpg.save("pipeline_controlnet_multi_call.npz", out)
    p2 = pipe((6, 7))
    for name, kw in error_cases(img, mask, pe, ne, ctls, H, W).items():
        try:
            p2(**kw)
            errors[name] = ["no error", ""]
        except Exception as e:  # noqa: BLE001  (recording whatever the reference raises is the point)
            errors[name] = [type(e).__name__, str(e)]
    import json

    out_dir = os.environ.get("PP_GOLDEN_OUT", mpg.HERE)
    with open(os.path.join(out_dir, "pipeline_controlnet_multi_errors.json"), "w") as f:
        json.dump(errors, f, indent=1, sort_keys=True)
    print("errors", errors)


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    main()
