"""`StableDiffusionControlNetInpaintPipeline` (PowerPaint v1 + ControlNet) — drop-in for the
reference class (powerpaint/pipelines/pipeline_PowerPaint_ControlNet.py:225; `__call__` :1347-1771).
The loop (:1663-1735: ControlNet on the 4-channel latents + control image, 9-channel UNet with the
12 down residuals + mid residual, CFG, scheduler.step) runs as one recorded CUDA program per step
(`FusedDenoiser(mode="controlnet")`); the t-independent `controlnet_cond_embedding(control_image)`
is evaluated once per call instead of once per step (SURVEY.md App. C (3)).

A list or tuple of ControlNets is wrapped in a `MultiControlNetModel` (:306): one control image, conditioning scale and
control_guidance window per net, residuals summed in net order inside the recorded step. `guess_mode` (or a ControlNet
whose config sets `global_pool_conditions`) runs the ControlNets on the conditional half of the CFG batch with
diffusers' logspace residual scales (:1669-1700).

Out of scope like upstream's dead code: `predict_woControl` (:996-1345, a buggy copy of the v1 `__call__`).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Union

import torch

from ..denoise import FusedDenoiser
from ..models.unet_2d_condition import ControlNetModel, MultiControlNetModel, UNet2DConditionModel
from .common import (StableDiffusionPipelineOutput, check_control_guidance, check_image, check_prompt_arguments,
                     decode_latents, prepare_mask_and_masked_image, preprocess_image, randn_tensor,
                     uint8_device_inputs)
from .pipeline_PowerPaint import StableDiffusionInpaintPipeline


class StableDiffusionControlNetInpaintPipeline(StableDiffusionInpaintPipeline):
    def __init__(self, vae, text_encoder, tokenizer, unet, controlnet, scheduler, safety_checker=None,
                 feature_extractor=None, requires_safety_checker: bool = False):
        super().__init__(vae, text_encoder, tokenizer, unet, scheduler, safety_checker, feature_extractor,
                         requires_safety_checker)
        if isinstance(controlnet, (list, tuple)):
            controlnet = MultiControlNetModel(controlnet)
        self.controlnet = controlnet
        self._denoiser_side = None

    def denoiser(self) -> FusedDenoiser:
        nets = self.controlnet.nets if isinstance(self.controlnet, MultiControlNetModel) else [self.controlnet]
        if not isinstance(self.unet, UNet2DConditionModel) or not all(isinstance(n, ControlNetModel) for n in nets):
            assert False, "unet / controlnet must be powerpaint_b200 UNet2DConditionModel / ControlNetModel(s)"
        if self._denoiser is None or self._denoiser_unet is not self.unet or self._denoiser_side is not self.controlnet:
            self._denoiser = FusedDenoiser(self.unet, self.controlnet, mode="controlnet")
            self._denoiser_unet, self._denoiser_side = self.unet, self.controlnet
        return self._denoiser

    def check_inputs_controlnet(self, prompt, image, height, width, callback_steps, negative_prompt=None,
                                prompt_embeds=None, negative_prompt_embeds=None, controlnet_conditioning_scale=1.0,
                                control_guidance_start=0.0, control_guidance_end=1.0):
        """the reference's `check_inputs` (:651-786; `image` = the control image) in its order, same exception types
        and messages. Unlike the v1 pipeline it does not look at `strength`."""
        if height % 8 != 0 or width % 8 != 0:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        if callback_steps is None or not isinstance(callback_steps, int) or callback_steps <= 0:
            raise ValueError(f"`callback_steps` has to be a positive integer but is {callback_steps} of type"
                             f" {type(callback_steps)}.")
        check_prompt_arguments(prompt, negative_prompt, prompt_embeds, negative_prompt_embeds)
        if isinstance(self.controlnet, ControlNetModel):
            check_image(image, prompt, prompt_embeds)
            if not isinstance(controlnet_conditioning_scale, float):
                raise TypeError("For single controlnet: `controlnet_conditioning_scale` must be type `float`.")
            check_control_guidance(control_guidance_start, control_guidance_end)
            return
        if not isinstance(self.controlnet, MultiControlNetModel):
            assert False
        n = len(self.controlnet.nets)
        if not isinstance(image, list):
            raise TypeError("For multiple controlnets: `image` must be type `list`")
        elif any(isinstance(i, list) for i in image):
            raise ValueError("A single batch of multiple conditionings are supported at the moment.")
        elif len(image) != n:
            raise ValueError(f"For multiple controlnets: `image` must have the same length as the number of "
                             f"controlnets, but got {len(image)} images and {n} ControlNets.")
        for image_ in image:
            check_image(image_, prompt, prompt_embeds)
        # (the reference's length check of a list scale is unreachable, :757-764: a shorter list runs fewer nets)
        if isinstance(controlnet_conditioning_scale, list):
            if any(isinstance(i, list) for i in controlnet_conditioning_scale):
                raise ValueError("A single batch of multiple conditionings are supported at the moment.")
        check_control_guidance(control_guidance_start, control_guidance_end, n)

    def check_image(self, image, prompt, prompt_embeds):
        """ref:pipeline_PowerPaint_ControlNet.py:788-827"""
        check_image(image, prompt, prompt_embeds)

    def _default_height_width(self, height, width, image):
        """missing sizes come from the init image, rounded down to a multiple of 8 (:914-937)"""
        while isinstance(image, list):
            image = image[0]
        if height is None:
            height = image.height if hasattr(image, "height") else image.shape[2]
            height = (height // 8) * 8
        if width is None:
            width = image.width if hasattr(image, "width") else image.shape[3]
            width = (width // 8) * 8
        return height, width

    def prepare_control_image(self, image, width, height, batch_size, num_images_per_prompt, device, dtype,
                              do_classifier_free_guidance=False, guess_mode=False):
        """control images are NOT normalised to [-1, 1] (do_normalize=False, :320-322)"""
        image = preprocess_image(image, height=height, width=width, do_normalize=False).to(dtype=torch.float32)
        repeat_by = batch_size if image.shape[0] == 1 else num_images_per_prompt
        image = image.repeat_interleave(repeat_by, dim=0).to(device=device, dtype=dtype)
        if do_classifier_free_guidance and not guess_mode:
            image = torch.cat([image] * 2)
        return image

    @torch.no_grad()
    def __call__(self, promptA: Union[str, List[str]] = None, promptB: Union[str, List[str]] = None, image=None,
                 mask=None, control_image=None, height: Optional[int] = None, width: Optional[int] = None,
                 strength: float = 1.0, tradoff: float = 1.0, tradoff_nag: float = 1.0, num_inference_steps: int = 50,
                 guidance_scale: float = 7.5, negative_promptA: Optional[Union[str, List[str]]] = None,
                 negative_promptB: Optional[Union[str, List[str]]] = None, num_images_per_prompt: Optional[int] = 1,
                 eta: float = 0.0, generator: Optional[Union[torch.Generator, List[torch.Generator]]] = None,
                 latents: Optional[torch.FloatTensor] = None, prompt_embeds: Optional[torch.FloatTensor] = None,
                 negative_prompt_embeds: Optional[torch.FloatTensor] = None, output_type: Optional[str] = "pil",
                 return_dict: bool = True, callback: Optional[Callable[[int, int, torch.FloatTensor], None]] = None,
                 callback_steps: int = 1, cross_attention_kwargs=None,
                 controlnet_conditioning_scale: Union[float, List[float]] = 0.5, guess_mode: bool = False,
                 control_guidance_start: Union[float, List[float]] = 0.0,
                 control_guidance_end: Union[float, List[float]] = 1.0):
        height, width = self._default_height_width(height, width, image)
        prompt, negative_prompt = promptA, negative_promptA
        multi = isinstance(self.controlnet, MultiControlNetModel)
        # align format for control guidance (:1491-1502), then the reference's checks (:1505-1517)
        if not isinstance(control_guidance_start, list) and isinstance(control_guidance_end, list):
            control_guidance_start = len(control_guidance_end) * [control_guidance_start]
        elif not isinstance(control_guidance_end, list) and isinstance(control_guidance_start, list):
            control_guidance_end = len(control_guidance_start) * [control_guidance_end]
        elif not isinstance(control_guidance_start, list) and not isinstance(control_guidance_end, list):
            mult = len(self.controlnet.nets) if multi else 1
            control_guidance_start, control_guidance_end = mult * [control_guidance_start], mult * [control_guidance_end]
        self.check_inputs_controlnet(prompt, control_image, height, width, callback_steps, negative_prompt,
                                     prompt_embeds, negative_prompt_embeds, controlnet_conditioning_scale,
                                     control_guidance_start, control_guidance_end)
        # valid for the reference, outside the hot path here
        if cross_attention_kwargs:
            raise NotImplementedError("cross_attention_kwargs (LoRA scale) is outside the hot path")
        if prompt is not None and isinstance(prompt, str):
            batch_size = 1
        elif prompt is not None and isinstance(prompt, list):
            batch_size = len(prompt)
        else:
            batch_size = prompt_embeds.shape[0]
        device = self._execution_device
        do_cfg = guidance_scale > 1.0
        if multi and isinstance(controlnet_conditioning_scale, float):
            controlnet_conditioning_scale = [controlnet_conditioning_scale] * len(self.controlnet.nets)
        guess_mode = guess_mode or self.controlnet.config.global_pool_conditions  # (:1536-1541)
        prompt_embeds = self._encode_prompt(promptA, promptB, tradoff, device, num_images_per_prompt, do_cfg,
                                            negative_promptA, negative_promptB, tradoff_nag,
                                            prompt_embeds=prompt_embeds, negative_prompt_embeds=negative_prompt_embeds)
        total = batch_size * num_images_per_prompt
        if multi:
            control = [self.prepare_control_image(c, width, height, total, num_images_per_prompt, device, torch.float32,
                                                  do_cfg, guess_mode) for c in control_image]
        else:
            control = self.prepare_control_image(control_image, width, height, total, num_images_per_prompt, device,
                                                 torch.float32, do_cfg, guess_mode)
        if uint8_device_inputs(self.vae, image, mask):  # see StableDiffusionInpaintPipeline.__call__
            if image.shape[-2:] != mask.shape[-2:] or image.shape[0] != mask.shape[0] or mask.shape[1] != 1:
                raise ValueError("uint8 image [B,3,H,W] and mask [B,1,H,W] must agree in batch and size")
            masked_image = init_image = image.contiguous()
        else:
            mask, masked_image, init_image = prepare_mask_and_masked_image(image, mask, height, width,
                                                                           return_image=True)
        self.scheduler.set_timesteps(num_inference_steps, device="cpu")
        timesteps, num_inference_steps = self.get_timesteps(num_inference_steps, strength, device)
        if self.unet.config.in_channels != 9:
            raise ValueError("the ControlNet inpainting path expects the 9-channel inpainting UNet")
        if num_inference_steps < 1:
            raise ValueError(f"After adjusting the num_inference_steps by strength parameter: {strength}, the number "
                             f"of pipeline steps is {num_inference_steps} which is < 1 and not appropriate for this "
                             "pipeline.")
        # strength < 1 (ref:pipeline_PowerPaint_ControlNet.py:1603-1625): noised image latents, shorter schedule
        latent_timestep = timesteps[:1].repeat(total)
        is_strength_max = strength == 1.0
        latents, noise = self.prepare_latents(total, self.vae.config.latent_channels, height, width, torch.float32,
                                              device, generator, latents, image=init_image,
                                              timestep=latent_timestep, is_strength_max=is_strength_max,
                                              return_noise=True, return_image_latents=False)
        mask, masked_image_latents = self.prepare_mask_latents(mask, masked_image, total, height, width, torch.float32,
                                                               device, generator, do_cfg)
        extra_step_kwargs = self.prepare_extra_step_kwargs(generator, eta)
        keep = [[1.0 - float(i / len(timesteps) < s or (i + 1) / len(timesteps) > e) for i in range(len(timesteps))]
                for s, e in zip(control_guidance_start, control_guidance_end)]
        # `controlnet_keep` (ref:pipeline_PowerPaint_ControlNet.py:1652-1658): the per-step scale
        # conditioning_scale * keep[i] of each net sits in the device side-scale table the recorded program indexes
        coef = self.scheduler.step_coefficients(timesteps, eta=extra_step_kwargs.get("eta", 0.0))
        ucoef = None
        if getattr(self.scheduler, "kind", "ddim") == "unipc":
            ucoef = self.scheduler.unipc_coefficients(first=len(self.scheduler.timesteps) - len(timesteps))
        noise_fn = None
        if eta > 0 and "eta" in extra_step_kwargs:  # schedulers without `eta` ignore it (signature sniffing, :536-551)
            shape = latents.shape

            def noise_fn(i):
                return randn_tensor(shape, generator=generator, device=device, dtype=torch.float32)
        cb = None
        if callback is not None:
            def cb(i, t, lat):
                if i % callback_steps == 0:
                    callback(i, t, lat)
                return None
        if multi:
            # MultiControlNetModel.forward zips images, scales and nets: a shorter scale list runs fewer nets
            n = min(len(control), len(controlnet_conditioning_scale))
            side = dict(control_image=control[:n], side_scale=[float(v) for v in controlnet_conditioning_scale[:n]],
                        side_keep=keep[:n])
        else:
            side = dict(control_image=control, side_scale=float(controlnet_conditioning_scale), side_keep=keep[0])
        if guess_mode:  # only passed when used: single-net callers see the keywords they always did
            side["guess_mode"] = True
        latents = self.denoiser().run(latents=latents, prompt_embeds=prompt_embeds, side_prompt_embeds=prompt_embeds,
                                      timesteps=timesteps, coef=coef, guidance_scale=guidance_scale,
                                      extra=torch.cat([mask, masked_image_latents], dim=1), **side,
                                      noise_fn=noise_fn, ucoef=ucoef, callback=cb)
        image_o = latents if output_type == "latent" else decode_latents(self.vae, latents, output_type)
        if not return_dict:
            return (image_o, None)
        return StableDiffusionPipelineOutput(images=image_o, nsfw_content_detected=None)
