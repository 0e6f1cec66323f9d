"""Calls of the ControlNet pipeline with several ControlNets and with guess mode, shared by the golden generator (which
records what the REFERENCE's `__call__` returns or raises) and the tests (which hold the product to it).

A case names the synthetic ControlNets it uses by their weight seeds: a tuple is passed to the pipeline as a list (the
pipeline wraps it in a MultiControlNetModel, one control image per net), an int as a single ControlNetModel."""
import torch

UNET_SEED = 5  # the 9-channel UNet of tests/golden/pipeline_controlnet_call.npz

CASES = {
    "two_nets": dict(nets=(6, 7), kw=dict(num_inference_steps=4, guidance_scale=7.5,
                                          controlnet_conditioning_scale=[0.5, 0.8], control_guidance_start=[0.0, 0.3],
                                          control_guidance_end=[1.0, 0.7])),
    # the reference's list-length check is unreachable: a 2-entry scale list runs the first two of three nets
    "three_nets_scale2": dict(nets=(6, 7, 8), kw=dict(num_inference_steps=3, guidance_scale=5.0,
                                                      controlnet_conditioning_scale=[0.6, 0.9])),
    "one_net_multi": dict(nets=(6,), kw=dict(num_inference_steps=3, guidance_scale=5.0,
                                             controlnet_conditioning_scale=0.5)),
    "guess_one": dict(nets=6, kw=dict(num_inference_steps=3, guidance_scale=7.5, controlnet_conditioning_scale=0.7,
                                      guess_mode=True)),
    "guess_two": dict(nets=(6, 7), kw=dict(num_inference_steps=3, guidance_scale=7.5,
                                           controlnet_conditioning_scale=0.6, control_guidance_end=[1.0, 0.5],
                                           guess_mode=True)),
    "guess_no_cfg": dict(nets=6, kw=dict(num_inference_steps=3, guidance_scale=1.0, controlnet_conditioning_scale=0.9,
                                         guess_mode=True)),
}

# GPU-sized calls (the latent size of GPU_CONTROLNET in pipeline_cases.py)
GPU_CASES = {
    "gpu_multi": dict(nets=(6, 7), size=64, seed=53, gen_seed=13,
                      kw=dict(num_inference_steps=6, guidance_scale=7.5, controlnet_conditioning_scale=[0.5, 0.7],
                              control_guidance_start=[0.0, 0.2], control_guidance_end=[0.7, 1.0])),
    "gpu_multi_guess": dict(nets=(6, 7), size=64, seed=53, gen_seed=13,
                            kw=dict(num_inference_steps=6, guidance_scale=7.5, controlnet_conditioning_scale=0.8,
                                    guess_mode=True)),
}


def control_images(n, batch, h, w, first=None):
    """one control image per net: net 0 gets `first` (or the image of pipeline_controlnet_call.npz's cases), net k > 0
    a seeded one of its own"""
    imgs = [first if first is not None else torch.rand(batch, 3, h, w, generator=torch.Generator().manual_seed(31))]
    for k in range(1, n):
        imgs.append(torch.rand(batch, 3, h, w, generator=torch.Generator().manual_seed(60 + k)))
    return imgs


def control_argument(nets, imgs):
    """the `control_image` keyword of a case: a list for a list of nets, the tensor for one net"""
    return list(imgs[:len(nets)]) if isinstance(nets, tuple) else imgs[0]


def error_cases(img, mask, pe, ne, ctls, H, W):
    """invalid calls with two ControlNets: name -> kwargs (ref:pipeline_PowerPaint_ControlNet.py:704-786)"""
    base = dict(image=img, mask=mask, control_image=list(ctls[:2]), prompt_embeds=pe, negative_prompt_embeds=ne,
                height=H, width=W, num_inference_steps=2, guidance_scale=7.5, output_type="latent", return_dict=False)

    def c(**kw):
        return {**base, **kw}

    return {
        "image_not_list": c(control_image=ctls[0]),
        "image_nested": c(control_image=[[ctls[0]], ctls[1]]),
        "image_count": c(control_image=[ctls[0]]),
        "scale_nested": c(controlnet_conditioning_scale=[[0.5], 0.5]),
        "guidance_start_count": c(control_guidance_start=[0.0, 0.1, 0.2]),
        "guidance_lengths_differ": c(control_guidance_start=[0.0, 0.1], control_guidance_end=[1.0]),
    }
