"""Generate tests/golden/unet_composition.npz from the REFERENCE's own model files.

    PP_REFERENCE_DIR=<checkout of the original PowerPaint project> python tests/golden/make_unet_golden.py

`powerpaint/models/{unet_2d_blocks,unet_2d_condition,BrushNet_CA}.py` of that checkout are imported UNMODIFIED; the absent
`diffusers` dependency is replaced by tests/golden/diffusers_shim (adapters over oracle/blocks.py for the primitive blocks
the SD-1.5 configuration instantiates, placeholders for everything else). What this pins is therefore the reference's
COMPOSITION — the 28 BrushNet add points and their pop(0) order, which states the skip tuple keeps, the up-path pops and
`upsample_size`, `BrushNetModel.from_unet`, the ControlNet residual entry points, the time-embedding plumbing — not the
arithmetic of the primitive blocks themselves (oracle/blocks.py stays "parity unpinned" for those).

Weights are the deterministic synthetic state dicts the tests use everywhere (powerpaint_b200.models.synthetic_state_dict:
same key set as the reference modules, checked below by a strict load), so the fixture holds only outputs.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(HERE, "diffusers_shim"), os.environ["PP_REFERENCE_DIR"], ROOT]

from powerpaint.models.BrushNet_CA import BrushNetModel as RefBrushNet  # noqa: E402  (the reference, unmodified)
from powerpaint.models.unet_2d_condition import UNet2DConditionModel as RefUNet  # noqa: E402

from powerpaint_b200.engine import NetConfig  # noqa: E402
from powerpaint_b200.models import synthetic_state_dict  # noqa: E402

BOC, HEADS, CROSS, GROUPS = (32, 64, 128, 128), 4, 64, 8  # == oracle UNetConfig.tiny


def ref_unet(in_channels):
    return RefUNet(sample_size=8, in_channels=in_channels, out_channels=4, block_out_channels=BOC, layers_per_block=2,
                   cross_attention_dim=CROSS, attention_head_dim=HEADS, norm_num_groups=GROUPS,
                   down_block_types=("CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "DownBlock2D"),
                   up_block_types=("UpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D")).eval()


def cfg(in_channels):
    return NetConfig(in_channels=in_channels, block_out_channels=BOC, attention_head_dim=HEADS, cross_attention_dim=CROSS,
                     norm_num_groups=GROUPS)


def inputs(seed, cin, h, w):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(2, cin, h, w, generator=g), torch.randn(2, 77, CROSS, generator=g),
            torch.randn(2, 5, h, w, generator=g))


@torch.no_grad()
def main():
    out = {}
    # ---- v1: 9-channel UNet, plain forward (also an odd latent size: upsample_size path)
    u9 = ref_unet(9)
    u9.load_state_dict(synthetic_state_dict(cfg(9), "unet", 1234), strict=True)
    for tag, (h, w) in {"8x8": (8, 8), "10x12": (10, 12)}.items():
        x, ctx, _ = inputs(11, 9, h, w)
        out[f"unet9_{tag}"] = u9(x, 321, ctx).sample.numpy()
    # two more seeds at another timestep, and the parameter names, that the oracle is held to
    for seed, (h, w) in ((3, (8, 8)), (4, (12, 10))):
        x, ctx, _ = inputs(seed, 9, h, w)
        out[f"unet9_seed{seed}_{h}x{w}"] = u9(x, 77, ctx).sample.numpy()
    out["unet9_state_dict_keys"] = np.array(sorted(u9.state_dict()))
    # ---- v2: BrushNet forward (28 outputs), 4-channel UNet consuming them, from_unet
    u4 = ref_unet(4)
    u4.load_state_dict(synthetic_state_dict(cfg(4), "unet", 1234), strict=True)
    bn = RefBrushNet.from_unet(u4, conditioning_channels=5).eval()
    fu = bn.state_dict()
    out["from_unet_conv_in_condition"] = fu["conv_in_condition.weight"].clone().numpy()  # (state_dict shares storage)
    out["from_unet_zero_conv_absmax"] = np.array([max(float(v.abs().max()) for k, v in fu.items() if k.startswith("brushnet_"))])
    out["from_unet_trunk_equal"] = np.array([int(all(torch.equal(fu[k], v) for k, v in u4.state_dict().items()
                                                      if k in fu and not k.startswith("conv_in")))])
    # from_unet makes conv_in_condition.bias THE SAME Parameter as unet.conv_in.bias (BrushNet_CA.py:530): loading other
    # weights into this object would overwrite the UNet's bias too, so the BrushNet that gets its own weights is a copy
    import copy
    bn = copy.deepcopy(bn)
    bn.load_state_dict(synthetic_state_dict(cfg(4), "brushnet", 77), strict=True)
    x, ctx, cond = inputs(13, 4, 8, 8)
    d, m, u = bn(x, 500, ctx, brushnet_cond=cond, conditioning_scale=0.8, return_dict=False)
    assert len(d) == 12 and len(u) == 15
    for i, t in enumerate(list(d) + [m] + list(u)):
        out[f"brushnet_{i:02d}"] = t.numpy()
    out["unet4_with_adds"] = u4(x, 500, ctx, down_block_add_samples=[t.clone() for t in d], mid_block_add_sample=m,
                                up_block_add_samples=[t.clone() for t in u]).sample.numpy()
    out["unet4_plain"] = u4(x, 500, ctx).sample.numpy()
    # ---- ControlNet-style residuals through the reference UNet (12 skip residuals + mid)
    g = torch.Generator().manual_seed(17)
    dres = tuple(torch.randn(t.shape, generator=g) * 0.1 for t in d)
    mres = torch.randn(m.shape, generator=g) * 0.1
    x9, ctx9, _ = inputs(19, 9, 8, 8)
    out["unet9_controlnet_residuals"] = u9(x9, 500, ctx9, down_block_additional_residuals=dres,
                                           mid_block_additional_residual=mres).sample.numpy()
    # the `config` surface of the reference classes (every constructor argument, unet_2d_condition.py:166-218,
    # BrushNet_CA.py:139-186), for the product's `.config.<name>` to be held to
    import json

    def plain(cfg):
        return {k: (list(v) if isinstance(v, tuple) else v) for k, v in dict(cfg).items()}

    with open(os.path.join(HERE, "model_configs.json"), "w") as f:
        json.dump({"unet9": plain(u9.config), "brushnet": plain(bn.config)}, f, indent=1, sort_keys=True)
    path = os.path.join(HERE, "unet_composition.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in list(out.items())[:4]}, "...", len(out), "arrays")


if __name__ == "__main__":
    main()
