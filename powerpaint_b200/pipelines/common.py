"""Host-side helpers shared by the three pipelines (pre/post-processing = SURVEY.md §8f "next"
rows; they run once per call outside the denoising loop and stay on PIL / torch for now).

Restated from the reference: `prepare_mask_and_masked_image`
(powerpaint/pipelines/pipeline_PowerPaint.py:39-153), diffusers `randn_tensor` and
`VaeImageProcessor` pre/post-processing (SURVEY.md App. A.10).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Union

import numpy as np
import PIL.Image
import torch


@dataclass
class StableDiffusionPipelineOutput:
    images: Union[List[PIL.Image.Image], np.ndarray, torch.Tensor]
    nsfw_content_detected: Optional[List[bool]]


def randn_tensor(shape, generator=None, device=None, dtype=None):
    """diffusers.utils.torch_utils.randn_tensor: a CPU generator with a CUDA target samples on the
    CPU and moves (so seeds are device independent); a list of generators samples per batch item."""
    device = torch.device(device) if device is not None else torch.device("cpu")
    batch = shape[0]
    rand_device = device
    if generator is not None:
        gen_dev = generator[0].device.type if isinstance(generator, list) else generator.device.type
        if gen_dev != device.type and gen_dev == "cpu":
            rand_device = torch.device("cpu")
        elif gen_dev != device.type and gen_dev == "cuda":
            raise ValueError(f"Cannot generate a {device} tensor from a generator of type {gen_dev}.")
    if isinstance(generator, list) and len(generator) == 1:
        generator = generator[0]
    if isinstance(generator, list):
        s = (1,) + tuple(shape[1:])
        lat = [torch.randn(s, generator=generator[i], device=rand_device, dtype=dtype) for i in range(batch)]
        return torch.cat(lat, dim=0).to(device)
    return torch.randn(shape, generator=generator, device=rand_device, dtype=dtype).to(device)


def prepare_mask_and_masked_image(image, mask, height, width, return_image: bool = False):
    """(mask [B,1,H,W] in {0,1}, masked_image [B,3,H,W] in [-1,1]) from PIL / numpy / tensor inputs;
    same accepted types, range checks and exceptions as the reference (:39-153)."""
    if image is None:
        raise ValueError("`image` input cannot be undefined.")
    if mask is None:
        raise ValueError("`mask_image` input cannot be undefined.")
    if isinstance(image, torch.Tensor):
        if not isinstance(mask, torch.Tensor):
            raise TypeError(f"`image` is a torch.Tensor but `mask` (type: {type(mask)} is not")
        # uint8 tensors (NCHW, any device) are the device-resident form of the uint8 numpy / PIL inputs the
        # reference converts with `/ 127.5 - 1` and `/ 255` (:123-140): < 1 MB per 512^2 image over PCIe, the
        # conversion runs where the tensor lives
        if image.dtype == torch.uint8:
            image = image.to(torch.float32) / 127.5 - 1.0
        if mask.dtype == torch.uint8:
            mask = mask.to(torch.float32) / 255.0
        if image.ndim == 3:
            assert image.shape[0] == 3, "Image outside a batch should be of shape (3, H, W)"
            image = image.unsqueeze(0)
        if mask.ndim == 2:
            mask = mask.unsqueeze(0).unsqueeze(0)
        if mask.ndim == 3:
            mask = mask.unsqueeze(0) if mask.shape[0] == 1 else mask.unsqueeze(1)
        assert image.ndim == 4 and mask.ndim == 4, "Image and Mask must have 4 dimensions"
        assert image.shape[-2:] == mask.shape[-2:], "Image and Mask must have the same spatial dimensions"
        assert image.shape[0] == mask.shape[0], "Image and Mask must have the same batch size"
        if image.min() < -1 or image.max() > 1:
            raise ValueError("Image should be in [-1, 1] range")
        if mask.min() < 0 or mask.max() > 1:
            raise ValueError("Mask should be in [0, 1] range")
        mask = mask.clone()
        mask[mask < 0.5] = 0
        mask[mask >= 0.5] = 1
        image = image.to(dtype=torch.float32)
    elif isinstance(mask, torch.Tensor):
        raise TypeError(f"`mask` is a torch.Tensor but `image` (type: {type(image)} is not")
    else:
        if isinstance(image, (PIL.Image.Image, np.ndarray)):
            image = [image]
        if isinstance(image, list) and isinstance(image[0], PIL.Image.Image):
            image = [i.resize((width, height), resample=PIL.Image.LANCZOS) for i in image]
            image = np.concatenate([np.array(i.convert("RGB"))[None, :] for i in image], axis=0)
        elif isinstance(image, list) and isinstance(image[0], np.ndarray):
            image = np.concatenate([i[None, :] for i in image], axis=0)
        image = torch.from_numpy(image.transpose(0, 3, 1, 2)).to(dtype=torch.float32) / 127.5 - 1.0
        if isinstance(mask, (PIL.Image.Image, np.ndarray)):
            mask = [mask]
        if isinstance(mask, list) and isinstance(mask[0], PIL.Image.Image):
            mask = [i.resize((width, height), resample=PIL.Image.LANCZOS) for i in mask]
            mask = np.concatenate([np.array(m.convert("L"))[None, None, :] for m in mask], axis=0)
            mask = mask.astype(np.float32) / 255.0
        elif isinstance(mask, list) and isinstance(mask[0], np.ndarray):
            mask = np.concatenate([m[None, None, :] for m in mask], axis=0)
        mask = mask.copy()
        mask[mask < 0.5] = 0
        mask[mask >= 0.5] = 1
        mask = torch.from_numpy(mask)
    masked_image = image * (mask < 0.5)
    if return_image:
        return mask, masked_image, image
    return mask, masked_image


_IMAGE_KINDS = ("one of PIL image, numpy array, torch tensor, list of PIL images, list of numpy arrays or list of torch "
                "tensors")


def _is_image_input(x) -> bool:
    one = (PIL.Image.Image, torch.Tensor, np.ndarray)
    return isinstance(x, one) or (isinstance(x, list) and len(x) > 0 and isinstance(x[0], one))


def check_image(image, prompt, prompt_embeds, mask=None, with_mask: bool = False):
    """`check_image` of the ControlNet / BrushNet pipelines (ref:pipeline_PowerPaint_ControlNet.py:788-827,
    ref:pipeline_PowerPaint_Brushnet_CA.py:868-922): accepted container types, then the image batch against the prompt
    batch — same exception types and messages."""
    if not _is_image_input(image):
        raise TypeError(f"image must be passed and be {_IMAGE_KINDS}, but is {type(image)}")
    if with_mask and not _is_image_input(mask):
        raise TypeError(f"mask must be passed and be {_IMAGE_KINDS}, but is {type(mask)}")
    image_batch_size = 1 if isinstance(image, PIL.Image.Image) else len(image)
    if prompt is not None and isinstance(prompt, str):
        prompt_batch_size = 1
    elif prompt is not None and isinstance(prompt, list):
        prompt_batch_size = len(prompt)
    else:
        prompt_batch_size = prompt_embeds.shape[0]
    if image_batch_size != 1 and image_batch_size != prompt_batch_size:
        raise ValueError("If image batch size is not 1, image batch size must be same as prompt batch size. image batch "
                         f"size: {image_batch_size}, prompt batch size: {prompt_batch_size}")


def check_prompt_arguments(prompt, negative_prompt, prompt_embeds, negative_prompt_embeds):
    """the prompt / embedding exclusivity rules every reference `check_inputs` shares
    (ref:pipeline_PowerPaint.py:575-602, ref:pipeline_PowerPaint_Brushnet_CA.py:782-807, ref:…ControlNet.py:675-700)"""
    if prompt is not None and prompt_embeds is not None:
        raise ValueError(f"Cannot forward both `prompt`: {prompt} and `prompt_embeds`: {prompt_embeds}. Please make "
                         "sure to only forward one of the two.")
    elif prompt is None and prompt_embeds is None:
        raise ValueError("Provide either `prompt` or `prompt_embeds`. Cannot leave both `prompt` and `prompt_embeds` "
                         "undefined.")
    elif prompt is not None and not isinstance(prompt, (str, list)):
        raise ValueError(f"`prompt` has to be of type `str` or `list` but is {type(prompt)}")
    if negative_prompt is not None and negative_prompt_embeds is not None:
        raise ValueError(f"Cannot forward both `negative_prompt`: {negative_prompt} and `negative_prompt_embeds`:"
                         f" {negative_prompt_embeds}. Please make sure to only forward one of the two.")
    if prompt_embeds is not None and negative_prompt_embeds is not None:
        if prompt_embeds.shape != negative_prompt_embeds.shape:
            raise ValueError("`prompt_embeds` and `negative_prompt_embeds` must have the same shape when passed "
                             f"directly, but got: `prompt_embeds` {prompt_embeds.shape} != "
                             f"`negative_prompt_embeds` {negative_prompt_embeds.shape}.")


def check_control_guidance(control_guidance_start, control_guidance_end, n_nets: Optional[int] = None):
    """ref:pipeline_PowerPaint_Brushnet_CA.py:836-855, ref:pipeline_PowerPaint_ControlNet.py:768-786; `n_nets`: the
    number of ControlNets of a MultiControlNetModel (one window per net)"""
    if len(control_guidance_start) != len(control_guidance_end):
        raise ValueError(f"`control_guidance_start` has {len(control_guidance_start)} elements, but "
                         f"`control_guidance_end` has {len(control_guidance_end)} elements. Make sure to provide the "
                         "same number of elements to each list.")
    if n_nets is not None and len(control_guidance_start) != n_nets:
        raise ValueError(f"`control_guidance_start`: {control_guidance_start} has {len(control_guidance_start)} elements "
                         f"but there are {n_nets} controlnets available. Make sure to provide {n_nets}.")
    for start, end in zip(control_guidance_start, control_guidance_end):
        if start >= end:
            raise ValueError(f"control guidance start: {start} cannot be larger or equal to control guidance end: "
                             f"{end}.")
        if start < 0.0:
            raise ValueError(f"control guidance start: {start} can't be smaller than 0.")
        if end > 1.0:
            raise ValueError(f"control guidance end: {end} can't be larger than 1.0.")


def preprocess_image(image, height=None, width=None, do_normalize=True) -> torch.Tensor:
    """VaeImageProcessor.preprocess: PIL/np/tensor -> float32 NCHW, resized (lanczos), [-1,1] if
    do_normalize (the control-image processor uses do_normalize=False,
    pipeline_PowerPaint_ControlNet.py:320-322)."""
    if isinstance(image, torch.Tensor):
        t = image if image.ndim == 4 else image.unsqueeze(0)
        if t.dtype == torch.uint8:  # device-resident form of a uint8 numpy / PIL input
            t = t.to(torch.float32) / 255.0
            return 2.0 * t - 1.0 if do_normalize else t
        t = t.to(torch.float32)
        if do_normalize and t.min() >= 0:
            t = 2.0 * t - 1.0
        return t
    if isinstance(image, (PIL.Image.Image, np.ndarray)):
        image = [image]
    if isinstance(image[0], PIL.Image.Image):
        if height is not None and width is not None:
            image = [i.resize((width, height), resample=PIL.Image.LANCZOS) for i in image]
        arr = np.stack([np.array(i.convert("RGB")).astype(np.float32) / 255.0 for i in image], axis=0)
    else:
        arr = np.stack([i.astype(np.float32) for i in image], axis=0)
        if arr.max() > 1.0:
            arr = arr / 255.0
    t = torch.from_numpy(arr.transpose(0, 3, 1, 2))
    return 2.0 * t - 1.0 if do_normalize else t


def postprocess_image(image: torch.Tensor, output_type: str = "pil", do_denormalize=None):
    """VaeImageProcessor.postprocess: (x/2+0.5).clamp(0,1) -> pt / np / pil"""
    if output_type == "latent":
        return image
    if do_denormalize is None:
        do_denormalize = [True] * image.shape[0]
    image = torch.stack([(image[i] / 2 + 0.5).clamp(0, 1) if do_denormalize[i] else image[i]
                         for i in range(image.shape[0])])
    if output_type == "pt":
        return image
    arr = image.detach().cpu().permute(0, 2, 3, 1).float().numpy()
    if output_type == "np":
        return arr
    if output_type == "pil":
        arr = (arr * 255).round().astype("uint8")
        return [PIL.Image.fromarray(a) for a in arr]
    raise ValueError(f"unsupported output_type {output_type}")


def decode_latents(vae, latents: torch.Tensor, output_type: str):
    """`vae.decode(latents / scaling_factor)` + `VaeImageProcessor.postprocess` (pipeline_PowerPaint.py:1051,:1062).
    With the kernel-backed AutoencoderKL the denormalisation (and for "pil" / "uint8" the x255 rounding) is fused
    into the pass that reads the decoded image; "uint8" (an extension: uint8 NHWC tensor left on the device, what
    "pil" images are built from) lets a serving loop gather / download 1 byte per channel."""
    z = latents / vae.config.scaling_factor
    if hasattr(vae, "decode_postprocessed"):
        if output_type in ("pil", "uint8"):
            u8 = vae.decode_postprocessed(z, uint8=True)
            if output_type == "uint8":
                return u8
            arr = u8.cpu().numpy()
            return [PIL.Image.fromarray(a) for a in arr]
        if output_type in ("pt", "np"):
            img = vae.decode_postprocessed(z, uint8=False)
            return img if output_type == "pt" else img.cpu().permute(0, 2, 3, 1).float().numpy()
        raise ValueError(f"unsupported output_type {output_type}")
    image = vae.decode(z.to(vae.dtype), return_dict=False)[0]
    if output_type == "uint8":
        image = postprocess_image(image.float(), output_type="pt")
        return (image * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    return postprocess_image(image.float(), output_type=output_type)


def uint8_device_inputs(vae, image, mask) -> bool:
    """uint8 CUDA image + mask tensors and a VAE that can read them directly (one fused pre-processing kernel)"""
    return (torch.is_tensor(image) and torch.is_tensor(mask) and image.dtype == torch.uint8 and image.is_cuda
            and mask.is_cuda and image.ndim == 4 and mask.ndim == 4 and hasattr(vae, "encode_uint8"))


def encode_text(tokenizer, text_encoder, prompts, device, max_length=None) -> torch.Tensor:
    """tokenize (max_length padding, truncation) + text encoder last hidden state"""
    max_length = max_length or tokenizer.model_max_length
    ids = tokenizer(prompts, padding="max_length", max_length=max_length, truncation=True,
                    return_tensors="pt").input_ids
    return text_encoder(ids.to(device))[0]


def vae_encode(vae, image: torch.Tensor, generator=None) -> torch.Tensor:
    """reference `_encode_vae_image` (pipeline_PowerPaint.py:657-669)"""
    image = image.to(getattr(vae, "dtype", image.dtype))
    if isinstance(generator, list):
        lat = [vae.encode(image[i:i + 1]).latent_dist.sample(generator=generator[i]) for i in range(image.shape[0])]
        lat = torch.cat(lat, dim=0)
    else:
        lat = vae.encode(image).latent_dist.sample(generator=generator)
    return vae.config.scaling_factor * lat.float()
