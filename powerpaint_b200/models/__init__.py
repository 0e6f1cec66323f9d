from .autoencoder_kl import AutoencoderKL
from .clip_text import CLIPTextModel
from .unet_2d_condition import (BrushNetModel, BrushNetOutput, ControlNetModel, ControlNetOutput,
                                MultiControlNetModel, UNet2DConditionModel, UNet2DConditionOutput)
from .spec import param_shapes, synthetic_state_dict

__all__ = ["AutoencoderKL", "BrushNetModel", "BrushNetOutput", "CLIPTextModel", "ControlNetModel", "ControlNetOutput",
           "MultiControlNetModel", "UNet2DConditionModel", "UNet2DConditionOutput", "param_shapes", "synthetic_state_dict"]
