"""The diffusers 0.27 behaviour the ControlNet golden of several nets and guess mode needs, on top of
tests/golden/diffusers_shim (used by make_controlnet_multi_golden.py only):

  ControlNetModel       the shim's oracle ControlNet, with diffusers' guess-mode residual scales
  MultiControlNetModel  diffusers' class: `.nets`, `dtype`, `config`, and a forward that zips images, scales and nets
                        (a shorter scale list runs fewer nets) and sums the residuals in net order

`install()` makes `diffusers.pipelines.controlnet.MultiControlNetModel` this class, also in the namespace of the
reference's pipeline_PowerPaint_ControlNet.py, which binds the name when it is imported (its package imports every
pipeline). The reference file itself is not changed."""
import torch
from diffusers.models import ControlNetModel as _ShimControlNetModel

from oracle.controlnet_multi import guess_scales
from oracle.unet import ControlNetOracle


class ControlNetModel(_ShimControlNetModel):
    def forward(self, sample, timestep, encoder_hidden_states, controlnet_cond, conditioning_scale=1.0,
                guess_mode=False, return_dict=True, **kw):
        down, mid = ControlNetOracle.forward(self, sample, timestep, encoder_hidden_states, controlnet_cond,
                                             1.0 if guess_mode else conditioning_scale)
        if guess_mode:
            down, mid = guess_scales(down, mid, conditioning_scale)
        return down, mid


class MultiControlNetModel(torch.nn.Module):
    def __init__(self, controlnets):
        super().__init__()
        self.nets = torch.nn.ModuleList(controlnets)

    @property
    def dtype(self):
        return self.nets[0].dtype

    @property
    def config(self):
        return self.nets[0].config

    def forward(self, sample, timestep, encoder_hidden_states, controlnet_cond, conditioning_scale, class_labels=None,
                timestep_cond=None, attention_mask=None, added_cond_kwargs=None, cross_attention_kwargs=None,
                guess_mode=False, return_dict=True):
        for i, (image, scale, controlnet) in enumerate(zip(controlnet_cond, conditioning_scale, self.nets)):
            down_samples, mid_sample = controlnet(sample=sample, timestep=timestep,
                                                  encoder_hidden_states=encoder_hidden_states, controlnet_cond=image,
                                                  conditioning_scale=scale, guess_mode=guess_mode,
                                                  return_dict=return_dict)
            if i == 0:
                down_block_res_samples, mid_block_res_sample = down_samples, mid_sample
            else:
                down_block_res_samples = [a + b for a, b in zip(down_block_res_samples, down_samples)]
                mid_block_res_sample += mid_sample
        return down_block_res_samples, mid_block_res_sample


def install():
    import diffusers.pipelines.controlnet as dpc
    import powerpaint.pipelines.pipeline_PowerPaint_ControlNet as ref

    dpc.MultiControlNetModel = ref.MultiControlNetModel = MultiControlNetModel
