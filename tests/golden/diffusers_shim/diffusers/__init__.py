"""Stand-in for `diffusers==0.27.0`, JUST ENOUGH for the reference's own model files
(`powerpaint/models/{unet_2d_blocks,unet_2d_condition,BrushNet_CA}.py`) and pipeline files
(`powerpaint/pipelines/pipeline_PowerPaint{,_Brushnet_CA,_ControlNet}.py`: DiffusionPipeline plumbing,
VaeImageProcessor for tensors, a DDIM scheduler / AutoencoderKL / ControlNetModel that are the oracle's) to import and run
UNMODIFIED on the CPU, so that golden vectors of the reference's *composition* can be generated here
(tests/golden/make_unet_golden.py): where BrushNet's 28 adds go, which skip the tuple keeps, how the up path pops,
what `from_unet` copies, how ControlNet residuals enter.

It is test infrastructure and NOT a re-implementation of diffusers: the primitive blocks it exposes under the diffusers
names (ResnetBlock2D, Transformer2DModel, Down/Upsample2D, Timesteps, TimestepEmbedding) are thin adapters over the
oracle's restatements (oracle/blocks.py: "PARITY UNPINNED" for their arithmetic), everything the hot path never
instantiates is a placeholder that raises when constructed. The real diffusers package is absent from this image and
cannot be installed (no network).
"""
__version__ = "0.27.0-shim"
from .models import AsymmetricAutoencoderKL  # noqa: E402,F401
