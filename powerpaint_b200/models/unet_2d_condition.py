"""Drop-in `UNet2DConditionModel` / `BrushNetModel` / `ControlNetModel` for the PowerPaint hot path.

Same names, `forward` arguments, return types and `.config` attributes as the reference classes
(powerpaint/models/unet_2d_condition.py:1040-1058 forward signature, :166 config;
powerpaint/models/BrushNet_CA.py:690-704 forward, :456-464 from_unet; diffusers ControlNetModel as
called at powerpaint/pipelines/pipeline_PowerPaint_ControlNet.py:1686-1694), but `forward` runs the
recorded CUDA program of `powerpaint_b200.engine.NetEngine` instead of ~800 eager library kernels.

Parameters live in an `nn.Module` tree whose `state_dict()` keys equal the diffusers names, so
`safetensors.torch.load_model(unet, "unet/unet.safetensors")` (reference app.py:111) and
`load_state_dict` work unchanged; the packed bf16 copies are rebuilt lazily after any load.

API conventions kept from the reference (SURVEY.md §8b): inputs are caller-owned NCHW tensors and
are never mutated; the BrushNet add *lists* are consumed with `pop(0)` exactly like the
reference does (unet_2d_condition.py:1223); outputs are fresh tensors in `self.dtype`.
"""
from __future__ import annotations

import os
from dataclasses import asdict, dataclass
from types import SimpleNamespace
from typing import Any, Dict, List, Optional, Tuple, Union

import torch
import torch.nn as nn

from .. import ops
from ..engine import NetConfig, NetEngine
from .spec import param_shapes, synthetic_state_dict


@dataclass
class UNet2DConditionOutput:
    sample: torch.Tensor = None


@dataclass
class BrushNetOutput:
    up_block_res_samples: Tuple[torch.Tensor]
    down_block_res_samples: Tuple[torch.Tensor]
    mid_block_res_sample: torch.Tensor


@dataclass
class ControlNetOutput:
    down_block_res_samples: Tuple[torch.Tensor]
    mid_block_res_sample: torch.Tensor


class _Config(SimpleNamespace):
    """attribute + mapping access like diffusers' FrozenDict config"""

    def __getitem__(self, k):
        return getattr(self, k)

    def __contains__(self, k):
        return hasattr(self, k)

    def get(self, k, default=None):
        return getattr(self, k, default)


def _make_config(cfg: NetConfig, **extra) -> _Config:
    d = asdict(cfg)
    d.update(dict(sample_size=extra.pop("sample_size", 64), time_cond_proj_dim=None, flip_sin_to_cos=True,
                  freq_shift=0, act_fn="silu", use_linear_projection=False, only_cross_attention=False,
                  num_attention_heads=None, class_embed_type=None, num_class_embeds=None,
                  upcast_attention=False, resnet_time_scale_shift="default", downsample_padding=1,
                  projection_class_embeddings_input_dim=None, mid_block_type="UNetMidBlock2DCrossAttn",
                  center_input_sample=False, addition_embed_type=None,
                  # the remaining constructor arguments of the reference class (unet_2d_condition.py:166-218) at the
                  # only values the hot path implements, so that `config.<name>` reads the same on both sides
                  addition_embed_type_num_heads=64, addition_time_embed_dim=None, attention_type="default",
                  class_embeddings_concat=False, conv_in_kernel=3, conv_out_kernel=3, cross_attention_norm=None,
                  dropout=0.0, dual_cross_attention=False, encoder_hid_dim=None, encoder_hid_dim_type=None,
                  mid_block_only_cross_attention=None, resnet_out_scale_factor=1.0, resnet_skip_time_act=False,
                  reverse_transformer_layers_per_block=None, time_embedding_act_fn=None, time_embedding_dim=None,
                  time_embedding_type="positional", timestep_post_act=None, transformer_layers_per_block=1))
    d.update(extra)
    return _Config(**d)


class _HotPathModel(nn.Module):
    KIND = "unet"

    def __init__(self, cfg: Optional[NetConfig] = None, sample_size: int = 64, **cfg_kwargs):
        super().__init__()
        if cfg is None:
            cfg = NetConfig(**cfg_kwargs)
        self._cfg = cfg
        self.config = _make_config(cfg, sample_size=sample_size)
        self._out_dtype = torch.float32
        for name, shape in param_shapes(cfg, self.KIND).items():
            self._register(name, torch.zeros(shape))
        self._engine: Optional[NetEngine] = None
        self._generation = 0  # bumped whenever the parameters change: recorded programs of older engines are stale
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate())

    # ---- parameter tree with diffusers names
    def _register(self, name: str, value: torch.Tensor):
        parts = name.split(".")
        mod = self
        for p in parts[:-1]:
            if not hasattr(mod, p):
                mod.add_module(p, nn.Module())
            mod = getattr(mod, p)
        mod.register_parameter(parts[-1], nn.Parameter(value, requires_grad=False))

    def _invalidate(self):
        self._engine = None
        self._generation += 1

    @property
    def generation(self) -> int:
        return self._generation

    def _apply(self, fn, *a, **k):  # .to() / .cuda() / .half() move parameters: repack lazily
        self._invalidate()
        return super()._apply(fn, *a, **k)

    @classmethod
    def from_state_dict(cls, cfg: NetConfig, state_dict: Dict[str, torch.Tensor], **kw):
        m = cls(cfg, **kw)
        m.load_state_dict(state_dict, strict=True)
        return m

    @classmethod
    def synthetic(cls, cfg: NetConfig, seed: int = 1234, **kw):
        return cls.from_state_dict(cfg, synthetic_state_dict(cfg, cls.KIND, seed), **kw)

    # ---- checkpoint directories in the diffusers layout (ref:app.py:121-123,141-147,165-171)
    @classmethod
    def from_config(cls, config, **kw):
        """a diffusers `config.json` dictionary (or another model's `.config`) -> an uninitialised model"""
        from ..loading import net_config_from_diffusers

        d = dict(vars(config)) if not isinstance(config, dict) else dict(config)
        return cls(net_config_from_diffusers(d, cls.KIND), sample_size=d.get("sample_size") or 64, **kw)

    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path, subfolder: Optional[str] = None, torch_dtype=None,
                        revision: Optional[str] = None, variant: Optional[str] = None, local_files_only: bool = False,
                        cache_dir: Optional[str] = None, **unused):
        """`ModelMixin.from_pretrained` for a local directory or a cached hub snapshot: `config.json` +
        `diffusion_pytorch_model[.variant].safetensors | .bin`, strict load, on the CPU. `torch_dtype` selects the
        dtype of returned tensors (compute is bf16 x bf16 -> fp32 whatever it says)."""
        from ..loading import load_json, load_weights, resolve_checkpoint_dir

        d = resolve_checkpoint_dir(pretrained_model_name_or_path, subfolder, revision, local_files_only, cache_dir)
        model = cls.from_config(load_json(d, "config.json"))
        model.load_state_dict(load_weights(d, variant), strict=True)
        if torch_dtype is not None:
            model.to(dtype=torch_dtype)
        return model

    def save_pretrained(self, save_directory, variant: Optional[str] = None, **unused):
        import json
        import os

        from ..loading import net_config_to_diffusers, save_weights

        os.makedirs(save_directory, exist_ok=True)
        with open(os.path.join(save_directory, "config.json"), "w") as f:
            json.dump(net_config_to_diffusers(self._cfg, self.KIND, self.config), f, indent=2, sort_keys=True)
        save_weights(self.state_dict(), save_directory, variant=variant)

    # ---- diffusers-like surface
    @property
    def dtype(self) -> torch.dtype:
        return self._out_dtype

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    def to(self, *args, **kwargs):
        # the reference app calls unet.to(dtype=fp16); compute is always bf16 x bf16 -> fp32 here,
        # the requested dtype only selects the dtype of returned tensors
        dtype = kwargs.get("dtype")
        for a in args:
            if isinstance(a, torch.dtype):
                dtype = a
        if dtype is not None:
            self._out_dtype = dtype
            kwargs.pop("dtype", None)
            args = tuple(a for a in args if not isinstance(a, torch.dtype))
            if not args and not kwargs:
                return self
        return super().to(*args, **kwargs)

    def engine(self) -> NetEngine:
        if self._engine is None:
            dev = self.device
            if dev.type != "cuda":
                raise RuntimeError(f"{type(self).__name__} must be on a CUDA device (got {dev}); "
                                   "the hot path has no CPU fallback")
            self._engine = NetEngine(self._cfg, {k: v for k, v in self.state_dict().items()}, self.KIND, dev)
        return self._engine

    # ---- shared helpers
    @staticmethod
    def _timesteps(timestep, nb: int, device) -> torch.Tensor:
        t = timestep
        if not torch.is_tensor(t):
            t = torch.tensor([float(t)], dtype=torch.float32, device=device)
        else:
            t = t.to(device=device, dtype=torch.float32).reshape(-1)
        if t.numel() == 1:
            t = t.expand(nb)
        if t.numel() != nb:
            raise ValueError(f"timestep has {t.numel()} entries for a batch of {nb}")
        return t.contiguous()

    def _load_inputs(self, plan, sample, timestep, encoder_hidden_states, extra_channels=None):
        nb, c, h, w = sample.shape
        x = sample if extra_channels is None else torch.cat([sample, extra_channels.to(sample.dtype)], dim=1)
        x_in = plan.inputs["x_in"]
        xn = ops.nchw_to_nhwc(x.float().contiguous(), x_in.shape[-1])
        x_in.copy_(xn.view_as(x_in))
        plan.inputs["timesteps"].copy_(self._timesteps(timestep, nb, sample.device))
        # the cross-attention K / V^T projections of the prompt are recomputed on every eager forward (32 tiny
        # GEMMs over [nb, 77, 768]): an address / version key is not a content identity — a new prompt tensor
        # commonly lands on the freed block of the previous one. The fused loop projects once per call.
        plan.inputs["ctx"].copy_(encoder_hidden_states.to(torch.bfloat16))
        plan.ctx_program.run()

    @staticmethod
    def _to_nchw(t: torch.Tensor, nb, h, w, dtype) -> torch.Tensor:
        c = t.shape[-1]
        return ops.nhwc_to_nchw(t.view(nb, h, w, c)).to(dtype)


class UNet2DConditionModel(_HotPathModel):
    KIND = "unet"

    @torch.no_grad()
    def forward(self, sample: torch.Tensor, timestep: Union[torch.Tensor, float, int],
                encoder_hidden_states: torch.Tensor, class_labels: Optional[torch.Tensor] = None,
                timestep_cond: Optional[torch.Tensor] = None, attention_mask: Optional[torch.Tensor] = None,
                cross_attention_kwargs: Optional[Dict[str, Any]] = None,
                added_cond_kwargs: Optional[Dict[str, torch.Tensor]] = None,
                down_block_additional_residuals: Optional[Tuple[torch.Tensor]] = None,
                mid_block_additional_residual: Optional[torch.Tensor] = None,
                down_intrablock_additional_residuals: Optional[Tuple[torch.Tensor]] = None,
                encoder_attention_mask: Optional[torch.Tensor] = None, return_dict: bool = True,
                down_block_add_samples: Optional[List[torch.Tensor]] = None,
                mid_block_add_sample: Optional[torch.Tensor] = None,
                up_block_add_samples: Optional[List[torch.Tensor]] = None):
        for name, v in (("class_labels", class_labels), ("timestep_cond", timestep_cond),
                        ("attention_mask", attention_mask), ("added_cond_kwargs", added_cond_kwargs),
                        ("down_intrablock_additional_residuals", down_intrablock_additional_residuals),
                        ("encoder_attention_mask", encoder_attention_mask)):
            if v is not None:
                raise NotImplementedError(f"`{name}` is outside the PowerPaint SD-1.5 hot path")
        if cross_attention_kwargs:
            raise NotImplementedError("cross_attention_kwargs (LoRA scale / GLIGEN) are outside the hot path")
        if sample.dim() != 4 or sample.shape[1] != self._cfg.in_channels:
            raise ValueError(f"sample must be [B, {self._cfg.in_channels}, H, W], got {tuple(sample.shape)}")
        nb, _, h, w = sample.shape
        is_brushnet = (down_block_add_samples is not None and mid_block_add_sample is not None
                       and up_block_add_samples is not None)
        is_controlnet = mid_block_additional_residual is not None and down_block_additional_residuals is not None
        with torch.cuda.device(self.device):  # launches go to the stream of the model's device
            return self._forward(sample, timestep, encoder_hidden_states, is_brushnet, is_controlnet,
                                 down_block_add_samples, mid_block_add_sample, up_block_add_samples,
                                 down_block_additional_residuals, mid_block_additional_residual, return_dict)

    def _forward(self, sample, timestep, encoder_hidden_states, is_brushnet, is_controlnet, down_block_add_samples,
                 mid_block_add_sample, up_block_add_samples, down_block_additional_residuals,
                 mid_block_additional_residual, return_dict):
        nb, _, h, w = sample.shape
        eng = self.engine()
        plan = eng.plan(nb, h, w, encoder_hidden_states.shape[1], with_brushnet_adds=is_brushnet,
                        with_controlnet_res=is_controlnet)
        self._load_inputs(plan, sample, timestep, encoder_hidden_states)
        if is_brushnet:
            nd, nu = len(plan.inputs["adds_down"]), len(plan.inputs["adds_up"])
            if len(down_block_add_samples) != nd or len(up_block_add_samples) != nu:
                raise ValueError(f"expected {nd} down / {nu} up add samples, got "
                                 f"{len(down_block_add_samples)} / {len(up_block_add_samples)}")
            # the reference consumes the lists with pop(0) (unet_2d_condition.py:1223,:1232-1253,:1316-1339)
            for dst in plan.inputs["adds_down"]:
                src = down_block_add_samples.pop(0)
                dst.copy_(ops.nchw_to_nhwc(src.float().contiguous()).view_as(dst))
            plan.inputs["add_mid"].copy_(
                ops.nchw_to_nhwc(mid_block_add_sample.float().contiguous()).view_as(plan.inputs["add_mid"]))
            for dst in plan.inputs["adds_up"]:
                src = up_block_add_samples.pop(0)
                dst.copy_(ops.nchw_to_nhwc(src.float().contiguous()).view_as(dst))
        if is_controlnet:
            if len(down_block_additional_residuals) != len(plan.inputs["cn_down"]):
                raise ValueError("wrong number of down_block_additional_residuals")
            for dst, src in zip(plan.inputs["cn_down"], down_block_additional_residuals):
                dst.copy_(ops.nchw_to_nhwc(src.float().contiguous()).view_as(dst))
            plan.inputs["cn_mid"].copy_(
                ops.nchw_to_nhwc(mid_block_additional_residual.float().contiguous()).view_as(plan.inputs["cn_mid"]))
        plan.program.launch()
        out = self._to_nchw(plan.outputs["eps"], nb, h, w, self.dtype)
        if not return_dict:
            return (out,)
        return UNet2DConditionOutput(sample=out)


class BrushNetModel(_HotPathModel):
    KIND = "brushnet"

    def __init__(self, cfg: Optional[NetConfig] = None, **kw):
        if cfg is None and "in_channels" not in kw:
            kw["in_channels"] = 4
        super().__init__(cfg, **kw)
        self.config.brushnet_conditioning_channel_order = "rgb"
        self.config.global_pool_conditions = False

    @classmethod
    def from_unet(cls, unet: UNet2DConditionModel, brushnet_conditioning_channel_order: str = "rgb",
                  conditioning_embedding_out_channels=(16, 32, 96, 256), load_weights_from_unet: bool = True,
                  conditioning_channels: int = 5):
        """reference BrushNet_CA.py:456-542: clone the trunk; conv_in weights go to input channels
        0:4 AND 4:8 of conv_in_condition, channel 8 (mask) stays zero; zero-convs stay zero."""
        cfg = NetConfig(**{**asdict(unet._cfg), "conditioning_channels": conditioning_channels})
        bn = cls(cfg, sample_size=unet.config.sample_size)
        if load_weights_from_unet:
            src = unet.state_dict()
            dst = bn.state_dict()
            new = {}
            for k, v in dst.items():
                if k == "conv_in_condition.weight":
                    w = torch.zeros_like(v)
                    w[:, :4] = src["conv_in.weight"]
                    w[:, 4:8] = src["conv_in.weight"]
                    new[k] = w
                elif k == "conv_in_condition.bias":
                    new[k] = src["conv_in.bias"].clone()
                elif k in src and src[k].shape == v.shape:
                    new[k] = src[k].clone()
                else:
                    new[k] = v  # zero-initialised 1x1 convs (zero_module, BrushNet_CA.py:955-958)
            bn.load_state_dict(new)
        bn.to(unet.device)
        bn._out_dtype = unet.dtype
        return bn

    @torch.no_grad()
    def forward(self, sample: torch.FloatTensor, timestep: Union[torch.Tensor, float, int],
                encoder_hidden_states: torch.Tensor, brushnet_cond: torch.FloatTensor,
                conditioning_scale: float = 1.0, class_labels: Optional[torch.Tensor] = None,
                timestep_cond: Optional[torch.Tensor] = None, attention_mask: Optional[torch.Tensor] = None,
                added_cond_kwargs: Optional[Dict[str, torch.Tensor]] = None,
                cross_attention_kwargs: Optional[Dict[str, Any]] = None, guess_mode: bool = False,
                return_dict: bool = True):
        if guess_mode:
            raise NotImplementedError("guess_mode is outside the PowerPaint hot path (unused by app.py)")
        for name, v in (("class_labels", class_labels), ("timestep_cond", timestep_cond),
                        ("attention_mask", attention_mask), ("added_cond_kwargs", added_cond_kwargs)):
            if v is not None:
                raise NotImplementedError(f"`{name}` is outside the PowerPaint SD-1.5 hot path")
        nb, _, h, w = sample.shape
        with torch.cuda.device(self.device):
            # one recorded program for every conditioning_scale: the zero-conv epilogues read it from a device scalar
            plan = self.engine().plan(nb, h, w, encoder_hidden_states.shape[1], brushnet_outputs=True)
            plan.scale_dev.fill_(float(conditioning_scale))
            self._load_inputs(plan, sample, timestep, encoder_hidden_states, extra_channels=brushnet_cond)
            plan.program.launch()
            shapes_d, shape_m, shapes_u = self.engine()._state_shapes(nb, h, w)
            down = [self._to_nchw(t, nb, s[1], s[2], self.dtype) for t, s in zip(plan.outputs["down"], shapes_d)]
            mid = self._to_nchw(plan.outputs["mid"], nb, shape_m[1], shape_m[2], self.dtype)
            up = [self._to_nchw(t, nb, s[1], s[2], self.dtype) for t, s in zip(plan.outputs["up"], shapes_u)]
        if not return_dict:
            return (down, mid, up)
        return BrushNetOutput(down_block_res_samples=down, mid_block_res_sample=mid, up_block_res_samples=up)


class ControlNetModel(_HotPathModel):
    KIND = "controlnet"

    def __init__(self, cfg: Optional[NetConfig] = None, **kw):
        if cfg is None and "in_channels" not in kw:
            kw["in_channels"] = 4
        super().__init__(cfg, **kw)
        self.config.global_pool_conditions = False

    @torch.no_grad()
    def forward(self, sample: torch.FloatTensor, timestep: Union[torch.Tensor, float, int],
                encoder_hidden_states: torch.Tensor, controlnet_cond: torch.FloatTensor,
                conditioning_scale: float = 1.0, class_labels: Optional[torch.Tensor] = None,
                timestep_cond: Optional[torch.Tensor] = None, attention_mask: Optional[torch.Tensor] = None,
                added_cond_kwargs: Optional[Dict[str, torch.Tensor]] = None,
                cross_attention_kwargs: Optional[Dict[str, Any]] = None, guess_mode: bool = False,
                return_dict: bool = True):
        """`guess_mode`: the 12 down residuals are scaled by torch.logspace(-1, 0, 13)[:12] and the mid residual by 1.0,
        each times `conditioning_scale` (diffusers ControlNetModel.forward); the factors are constants of a plan
        recorded for guess mode, the scale stays a device scalar."""
        nb, _, h, w = sample.shape
        with torch.cuda.device(self.device):
            outs = self._run(sample, timestep, encoder_hidden_states, controlnet_cond, conditioning_scale, guess_mode)
            down, mid = self._residuals_nchw(outs, nb, h, w)
        if not return_dict:
            return (down, mid)
        return ControlNetOutput(down_block_res_samples=down, mid_block_res_sample=mid)

    def _run(self, sample, timestep, encoder_hidden_states, controlnet_cond, conditioning_scale, guess_mode):
        """one forward on the recorded plan: (down, mid) channels-last bf16 residuals owned by the plan"""
        nb, _, h, w = sample.shape
        if tuple(controlnet_cond.shape[2:]) != (8 * h, 8 * w):
            raise ValueError("controlnet_cond must be 8x the latent resolution")
        eng = self.engine()
        plan = eng.plan(nb, h, w, encoder_hidden_states.shape[1], guess_mode=bool(guess_mode))
        # t-independent (SURVEY.md App. C (3)): the 8-conv embedding is re-run only when the staged control
        # image actually differs (content comparison on the device; an address is not an identity)
        ci = plan.inputs["cond_in"]
        new_ci = ops.nchw_to_nhwc(controlnet_cond.float().contiguous(), ci.shape[-1]).view_as(ci)
        if not plan.outputs.get("cond_valid") or not torch.equal(new_ci, ci):
            ci.copy_(new_ci)
            plan.cond_program.run()
            plan.outputs["cond_valid"] = True
        plan.scale_dev.fill_(float(conditioning_scale))
        self._load_inputs(plan, sample, timestep, encoder_hidden_states)
        plan.program.launch()
        return plan.outputs["down"], plan.outputs["mid"]

    def _residuals_nchw(self, outs, nb, h, w):
        shapes_d, shape_m, _ = self.engine()._state_shapes(nb, h, w)
        down = [self._to_nchw(t, nb, sh[1], sh[2], self.dtype) for t, sh in zip(outs[0], shapes_d)]
        return down, self._to_nchw(outs[1], nb, shape_m[1], shape_m[2], self.dtype)


class MultiControlNetModel(nn.Module):
    """diffusers' `MultiControlNetModel`: several ControlNets whose residuals are summed (net 0 first). The reference
    pipeline wraps a list / tuple of ControlNets in it (ref:pipeline_PowerPaint_ControlNet.py:306)."""

    def __init__(self, controlnets):
        super().__init__()
        self.nets = nn.ModuleList(controlnets)

    @property
    def config(self):
        return self.nets[0].config

    @property
    def generation(self) -> tuple:
        """changes whenever the parameters of any net change"""
        return tuple(n.generation for n in self.nets)

    @property
    def dtype(self) -> torch.dtype:
        return self.nets[0].dtype

    @property
    def device(self) -> torch.device:
        return self.nets[0].device

    def to(self, *args, **kwargs):
        for n in self.nets:
            n.to(*args, **kwargs)
        return self

    @torch.no_grad()
    def forward(self, sample: torch.FloatTensor, timestep: Union[torch.Tensor, float, int],
                encoder_hidden_states: torch.Tensor, controlnet_cond: List[torch.Tensor],
                conditioning_scale: List[float], class_labels: Optional[torch.Tensor] = None,
                timestep_cond: Optional[torch.Tensor] = None, attention_mask: Optional[torch.Tensor] = None,
                added_cond_kwargs: Optional[Dict[str, torch.Tensor]] = None,
                cross_attention_kwargs: Optional[Dict[str, Any]] = None, guess_mode: bool = False,
                return_dict: bool = True):
        """zips images, scales and nets like diffusers (a shorter list runs fewer nets); returns (down, mid)"""
        for name, v in (("class_labels", class_labels), ("timestep_cond", timestep_cond),
                        ("attention_mask", attention_mask), ("added_cond_kwargs", added_cond_kwargs)):
            if v is not None:
                raise NotImplementedError(f"`{name}` is outside the PowerPaint SD-1.5 hot path")
        if cross_attention_kwargs:
            raise NotImplementedError("cross_attention_kwargs are outside the hot path")
        nb, _, h, w = sample.shape
        total = None
        with torch.cuda.device(self.device):
            for image, scale, net in zip(controlnet_cond, conditioning_scale, self.nets):
                d, m = net._run(sample, timestep, encoder_hidden_states, image, scale, guess_mode)
                if total is None:  # the plan owns its outputs: the sum lives in buffers of its own
                    total = ([t.clone() for t in d], m.clone())
                else:  # bf16 + bf16 -> bf16, the rounding of the fused loop's chained zero-convs
                    for acc, t in zip(total[0], d):
                        ops.add(acc, t, acc)
                    ops.add(total[1], m, total[1])
            if total is None:
                raise ValueError("no ControlNet ran: controlnet_cond / conditioning_scale are empty")
            return self.nets[0]._residuals_nchw(total, nb, h, w)

    def save_pretrained(self, save_directory, **kwargs):
        """net k goes to `save_directory` + ("" if k == 0 else f"_{k}") (diffusers layout)"""
        save_directory = os.fspath(save_directory)
        for k, net in enumerate(self.nets):
            net.save_pretrained(save_directory + ("" if k == 0 else f"_{k}"), **kwargs)

    @classmethod
    def from_pretrained(cls, pretrained_model_path, **kwargs):
        """loads `path`, `path_1`, `path_2`, ... until one is missing"""
        pretrained_model_path = os.fspath(pretrained_model_path)
        nets, k, path = [], 0, pretrained_model_path
        while os.path.isdir(path):
            nets.append(ControlNetModel.from_pretrained(path, **kwargs))
            k += 1
            path = pretrained_model_path + f"_{k}"
        if not nets:
            raise ValueError(f"No ControlNets found under {os.path.dirname(pretrained_model_path)}. Expected at least "
                             f"{pretrained_model_path + '_0'}.")
        return cls(nets)
