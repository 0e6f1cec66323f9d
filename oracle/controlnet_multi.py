"""ORACLE (test infrastructure, not product): several ControlNets and ControlNet guess mode in plain fp32 PyTorch.

  guess mode    diffusers ControlNetModel.forward: without global pooling the 12 down residuals are scaled by
                torch.logspace(-1, 0, 13)[:12] x conditioning_scale and the mid residual by 1.0 x conditioning_scale
  several nets  diffusers MultiControlNetModel.forward: the nets' residuals summed in net order
  the loop      powerpaint/pipelines/pipeline_PowerPaint_ControlNet.py:1663-1735 with a list of ControlNets and
                guess mode (:1669-1700)

PINNED for what the reference's own pipeline file decides: tests/golden/pipeline_controlnet_multi_call.npz (generator
tests/golden/make_controlnet_multi_golden.py).
"""
from __future__ import annotations

import torch

from .ddim import DDIMOracle


def guess_scales(down, mid, conditioning_scale: float):
    """diffusers' guess-mode factors applied to residuals computed at conditioning_scale 1.0"""
    scales = torch.logspace(-1, 0, len(down) + 1, device=mid.device) * conditioning_scale
    return [d * s for d, s in zip(down, scales)], mid * scales[-1]


def controlnet_forward(net, sample, timestep, encoder_hidden_states, controlnet_cond, conditioning_scale: float = 1.0,
                       guess_mode: bool = False):
    """`net` = oracle.unet.ControlNetOracle; (down list, mid) with diffusers' guess-mode scales when asked"""
    if not guess_mode:
        return net(sample, timestep, encoder_hidden_states, controlnet_cond, conditioning_scale)
    down, mid = net(sample, timestep, encoder_hidden_states, controlnet_cond, 1.0)
    return guess_scales(down, mid, conditioning_scale)


@torch.no_grad()
def loop_controlnet_multi(unet, controlnets, sched: DDIMOracle, latents, prompt_embeds, mask, masked_image_latents,
                          control_images, guidance_scale: float, conditioning_scales, keeps=None,
                          guess_mode: bool = False, record=None):
    """control_images[k] is [2B,3,H,W] (duplicated for CFG) or, in guess mode, [B,3,H,W]; keeps[k][i] =
    `controlnet_keep[i][k]` (or None for always kept). Guess mode with CFG runs the nets on the conditional half
    (latents, the second half of prompt_embeds) and pads their residuals with zeros for the unconditional half."""
    do_cfg = guidance_scale > 1.0
    half = guess_mode and do_cfg
    if do_cfg:
        mask = torch.cat([mask] * 2)
        masked_image_latents = torch.cat([masked_image_latents] * 2)
    for i, t in enumerate(sched.timesteps):
        x4 = torch.cat([latents] * 2) if do_cfg else latents
        xc, pc = (latents, prompt_embeds.chunk(2)[1]) if half else (x4, prompt_embeds)
        d = m = None
        for k, (net, img, s) in enumerate(zip(controlnets, control_images, conditioning_scales)):
            kp = keeps[k] if keeps is not None else None
            dk, mk = controlnet_forward(net, xc, int(t), pc, img, s * (kp[i] if kp is not None else 1.0), guess_mode)
            d, m = (dk, mk) if d is None else ([a + b for a, b in zip(d, dk)], m + mk)
        if half:
            d = [torch.cat([torch.zeros_like(r), r]) for r in d]
            m = torch.cat([torch.zeros_like(m), m])
        x9 = torch.cat([x4, mask, masked_image_latents], dim=1)
        eps = unet(x9, int(t), prompt_embeds, down_block_additional_residuals=d, mid_block_additional_residual=m)
        if do_cfg:
            a, c = eps.chunk(2)
            eps = a + guidance_scale * (c - a)
        latents = sched.step(eps, int(t), latents)
        if record is not None:
            record.append(latents.clone())
    return latents
