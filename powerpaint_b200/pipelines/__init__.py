from .pipeline_PowerPaint import StableDiffusionInpaintPipeline
from .pipeline_PowerPaint_Brushnet_CA import StableDiffusionPowerPaintBrushNetPipeline
from .pipeline_PowerPaint_ControlNet import StableDiffusionControlNetInpaintPipeline
from ..models.unet_2d_condition import MultiControlNetModel

__all__ = ["StableDiffusionInpaintPipeline", "StableDiffusionPowerPaintBrushNetPipeline",
           "StableDiffusionControlNetInpaintPipeline", "MultiControlNetModel"]
