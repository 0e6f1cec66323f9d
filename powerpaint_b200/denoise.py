"""The fused denoising loop: one recorded CUDA program per step, replayed as a CUDA graph.

Replaces the body of the reference loops
  v1          powerpaint/pipelines/pipeline_PowerPaint.py:988-1035
  v2 BrushNet powerpaint/pipelines/pipeline_PowerPaint_Brushnet_CA.py:1384-1449
  ControlNet  powerpaint/pipelines/pipeline_PowerPaint_ControlNet.py:1663-1735
i.e. per step: CFG duplication + channel concat -> [BrushNet | ControlNet] -> UNet -> CFG combine ->
DDIMScheduler.step. Here the step is a single `pp_program`:

    [side net forward]  ->  UNet forward (side-net residuals ride the UNet epilogues)
                        ->  pp_cfg_ddim_step: eps = u + s (c - u); x_{t-1}; writes the NEXT step's
                            bf16 channels-last net input for both CFG halves; bumps the step counter

The per-step scalars (timestep, DDIM coefficients, guidance scale) live in device tables indexed
by a device-side step counter, so one captured graph serves all steps; nothing crosses PCIe
inside the loop (the reference uploads `t` every step, unet_2d_condition.py:926). Step-invariant
work is hoisted: cross-attention K/V of the prompt(s), ControlNet's conditioning embedding, and
the constant input channels (mask, masked-image latents, BrushNet condition) are converted once.

All nets read ONE shared input buffer [n, h*w, 16]: channels 0..3 = latents, 4.. = the constant
channels of whichever net consumes them; nets that do not consume a channel carry zero weights
for it (weights are zero-padded at pack time), so no per-net concat exists. The constant channels are
written once per call; the step kernel only refreshes the four latent channels.

Per-step coefficient row (8 floats, `coef[step]`): 0-4 DDIM (sqrt(a_t), sqrt(1-a_t), sqrt(a_prev),
sqrt(1-a_prev-sigma^2), sigma), 5 guidance scale, 6 unused, 7 blend sqrt(a_t). The side nets' conditioning scales sit
in their own table `side_scale[step, k]` (n_side floats per step, k = side net): conditioning scale of net k x its keep
flag of the step (`brushnet_keep` / `controlnet_keep`, Brushnet_CA.py:1369-1376,1403-1409, ControlNet.py:1652-1658).
Net k's zero-conv epilogues multiply by entry k of the row the step counter selects, so a recorded plan serves every
guidance / conditioning scale and every control_guidance window.

Several ControlNets (`MultiControlNetModel`) record one after the other into the step program; net k's zero-convs add
net k-1's residuals as they store their own, so the last net's outputs hold the sum the UNet reads (net 0 first, as
diffusers sums them). In guess mode with CFG the ControlNets run on the conditional half only: batch B on the view
x_in[B:2B], writing the second half of [2B, ...] residual buffers whose first half stays zero.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Callable, Optional, Sequence

import torch

from . import ops
from .engine import NetEngine, Plan

MAX_STEPS = 1000
X_IN_C = 16
COEF_GUIDANCE = 5


class FusedDenoiser:
    """mode: 'v1' (UNet, 9-ch), 'brushnet' (BrushNet + 4-ch UNet), 'controlnet' (ControlNet or MultiControlNetModel +
    9-ch UNet)"""

    def __init__(self, unet, side=None, mode: str = "v1"):
        if mode not in ("v1", "brushnet", "controlnet"):
            raise ValueError(mode)
        if (mode == "v1") != (side is None):
            raise ValueError("side net must be given exactly for modes 'brushnet' / 'controlnet'")
        self.unet = unet
        self.side = side
        self.mode = mode
        # recorded plans, least recently used first; a plan owns its activation pool (a few GB at C2), so only
        # MAX_PLANS shapes are kept
        self._cache: "OrderedDict[tuple, dict]" = OrderedDict()
        self._stream: Optional[torch.cuda.Stream] = None

    MAX_PLANS = 2

    # ------------------------------------------------------------------ plan
    def _side_nets(self) -> list:
        """the side nets in summation order (a MultiControlNetModel's `.nets`, else the one side net)"""
        if self.side is None:
            return []
        return list(self.side.nets) if hasattr(self.side, "nets") else [self.side]

    def _get(self, B: int, h: int, w: int, do_cfg: bool, ctx_len: int, with_noise: bool,
             extra_per_copy: bool, sched: str = "ddim", blend: bool = False, n_side: int = 1,
             guess: bool = False) -> dict:
        # the key carries the parameter generation of each model: `load_state_dict` / `.to()` invalidate it,
        # and the cached entry keeps its engines alive, so a recycled id() can never alias a stale program
        nets = self._side_nets()[:n_side]
        key = (B, h, w, do_cfg, ctx_len, with_noise, extra_per_copy, sched, blend, n_side, guess, self.unet.generation,
               tuple(n.generation for n in nets))
        st = self._cache.get(key)
        if st is not None:
            self._cache.move_to_end(key)
            return st
        gens = tuple(n.generation for n in self._side_nets())
        for k in [k for k in self._cache if k[-2] != key[-2] or k[-1] != gens[:len(k[-1])]]:
            del self._cache[k]  # plans recorded against replaced weights
        while len(self._cache) >= self.MAX_PLANS:
            self._cache.popitem(last=False)
        dev = self.unet.device
        nb = 2 * B if do_cfg else B
        ue: NetEngine = self.unet.engine()
        prog, ctxprog = ops.Program(), ops.Program()
        x_in = torch.zeros(nb, h * w, X_IN_C, dtype=torch.bfloat16, device=dev)
        timesteps = torch.zeros(MAX_STEPS, dtype=torch.float32, device=dev)
        step_idx = torch.zeros(1, dtype=torch.int32, device=dev)
        coef = torch.zeros(MAX_STEPS, 8, dtype=torch.float32, device=dev)
        side_scale = torch.zeros(MAX_STEPS, max(n_side, 1), dtype=torch.float32, device=dev)
        pool = Plan()  # the nets of one step share one activation pool
        shared = dict(program=prog, ctx_program=ctxprog, x_in=x_in, timesteps=timesteps, step_idx=step_idx, pool=pool,
                      scale_dev=(side_scale[:, 0], step_idx, n_side))
        engines = [n.engine() for n in nets]
        st = dict(B=B, nb=nb, h=h, w=w, do_cfg=do_cfg, x_in=x_in, timesteps=timesteps, step_idx=step_idx, coef=coef,
                  side_scale=side_scale, program=prog, ctx_program=ctxprog, graph=False, with_noise=with_noise,
                  extra_per_copy=extra_per_copy, guess=guess, engines=(ue, *engines))
        side_plans = []
        if self.mode == "brushnet":
            se: NetEngine = engines[0]
            side_plan = se._build_plan(nb, h, w, ctx_len, False, False, True, 0, shared=shared)
            se.append_brushnet_outputs(side_plan, 1.0, scale_dev=shared["scale_dev"])
            side_plans.append(side_plan)
            shared_u = dict(shared, adds=(side_plan.outputs["down"], side_plan.outputs["mid"], side_plan.outputs["up"]))
            uplan = ue._build_plan(nb, h, w, ctx_len, True, False, True, 0, shared=shared_u)
        elif self.mode == "controlnet":
            half = guess and do_cfg  # ControlNets see the conditional half only
            nbc = B if half else nb
            res = None  # (down list, mid) of the previous net
            for k, se in enumerate(engines):
                sh = dict(shared, x_in=x_in[B:] if half else x_in, scale_dev=(side_scale[:, k], step_idx, n_side),
                          cn_res2=res)
                if guess:
                    sh["cn_alpha"] = se.guess_alphas()
                if half and k == len(engines) - 1:
                    # the UNet reads [2B, ...] residuals whose unconditional half is zero (torch.zeros_like, :1697-1700)
                    shapes_d, shape_m, _ = se._state_shapes(nb, h, w)
                    full_d = [torch.zeros(nb * hh * ww, c, dtype=torch.bfloat16, device=dev) for c, hh, ww in shapes_d]
                    full_m = torch.zeros(nb * shape_m[1] * shape_m[2], shape_m[0], dtype=torch.bfloat16, device=dev)
                    st["guess_residuals"] = (full_d, full_m)
                    sh["cn_out"] = ([t[t.shape[0] // 2:] for t in full_d], full_m[full_m.shape[0] // 2:])
                side_plan = se._build_plan(nbc, h, w, ctx_len, False, False, True, 0, shared=sh)
                side_plans.append(side_plan)
                res = (side_plan.outputs["down"], side_plan.outputs["mid"])
            if half:
                res = st["guess_residuals"]
            shared_u = dict(shared, cn=res)
            uplan = ue._build_plan(nb, h, w, ctx_len, False, True, True, 0, shared=shared_u)
        else:
            uplan = ue._build_plan(nb, h, w, ctx_len, False, False, True, 0, shared=shared)
        st["uplan"], st["side_plans"] = uplan, side_plans
        # fp32 master latents and the constant channels (channels-last)
        n_extra = nb if extra_per_copy else B
        st["latents"] = torch.zeros(B, h * w, 4, dtype=torch.float32, device=dev)
        st["extra"] = torch.zeros(n_extra, h * w, 5, dtype=torch.float32, device=dev)
        st["noise"] = torch.zeros(B, h * w, 4, dtype=torch.float32, device=dev)
        if sched == "unipc":
            # UniPCMultistepScheduler (the v2 app's scheduler, app.py:197): multistep state lives next to the latents
            for k in ("last_sample", "m1", "m2"):
                st[k] = torch.zeros(B, h * w, 4, dtype=torch.float32, device=dev)
            st["ucoef"] = torch.zeros(MAX_STEPS, 12, dtype=torch.float32, device=dev)
            prog.add(ops.unipc_desc(eps=uplan.outputs["eps"], eps_fp32=True, eps_ld=4, latents=st["latents"],
                                    last_sample=st["last_sample"], m1=st["m1"], m2=st["m2"], coef=coef,
                                    ucoef=st["ucoef"], step_idx=step_idx, advance_step=True, do_cfg=do_cfg, batch=B,
                                    hw=h * w, next_in=x_in, next_c=X_IN_C, n_copies=2 if do_cfg else 1))
        else:
            if blend:  # 4-channel UNet: known region kept on the noised original after every step
                st["blend_x0"] = torch.zeros(h * w, 4, dtype=torch.float32, device=dev)
                st["blend_mask"] = torch.zeros(h * w, dtype=torch.float32, device=dev)
                st["blend_noise"] = torch.zeros(B, h * w, 4, dtype=torch.float32, device=dev)
            prog.add(ops.cfg_ddim_desc(eps=uplan.outputs["eps"], eps_fp32=True, eps_ld=4, latents=st["latents"],
                                       coef=coef, step_idx=step_idx, advance_step=True,
                                       noise=st["noise"] if with_noise else None, guidance_scale=0.0,
                                       guidance_from_coef=True, do_cfg=do_cfg, batch=B, hw=h * w, next_in=x_in,
                                       next_c=X_IN_C, n_copies=2 if do_cfg else 1, extra=None, extra_c=0,
                                       blend_x0=st.get("blend_x0"), blend_mask=st.get("blend_mask"),
                                       blend_noise=st.get("blend_noise")))
        st["bytes"] = uplan.bytes + sum(p.bytes for p in side_plans)
        self._cache[key] = st
        return st

    @property
    def launches_per_step(self) -> int:
        return max((s["program"].num_launches for s in self._cache.values()), default=0)

    # ------------------------------------------------------------------ run
    def _fill_x_in(self, st: dict, latents_only: bool = False):
        B, do_cfg, x_in = st["B"], st["do_cfg"], st["x_in"]
        lat16 = st["latents"].to(torch.bfloat16)
        for cpy in range(2 if do_cfg else 1):
            x_in[cpy * B:(cpy + 1) * B, :, :4] = lat16
            if not latents_only:
                ex = st["extra"][cpy * B:(cpy + 1) * B] if st["extra_per_copy"] else st["extra"]
                x_in[cpy * B:(cpy + 1) * B, :, 4:9] = ex.to(torch.bfloat16)

    @torch.no_grad()
    def run(self, *, latents: torch.Tensor, prompt_embeds: torch.Tensor, timesteps, coef: torch.Tensor,
            guidance_scale: float, extra: Optional[torch.Tensor] = None,
            side_prompt_embeds: Optional[torch.Tensor] = None, control_image=None,
            side_scale=1.0, side_keep: Optional[Sequence] = None,
            noise_fn: Optional[Callable[[int], torch.Tensor]] = None, ucoef: Optional[torch.Tensor] = None,
            blend: Optional[dict] = None,
            callback: Optional[Callable[[int, int, torch.Tensor], Optional[torch.Tensor]]] = None,
            use_graph: bool = True, guess_mode: bool = False) -> torch.Tensor:
        """latents [B,4,h,w]; prompt_embeds [nb,77,768] for the UNet (negative half first when CFG);
        extra [B or nb,5,h,w] = constant channels (v1/controlnet: mask + masked-image latents;
        brushnet: conditioning latents + mask; nb rows = one set per CFG half); side_prompt_embeds
        for the side net; `side_scale` x `side_keep[i]` (default 1) scales the side net's residuals at step i.
        Several ControlNets (a MultiControlNetModel side): `control_image`, `side_scale` and `side_keep` are lists with
        one entry per net (`side_keep[k][i]`); a list shorter than `.nets` runs the first len(list) nets. `guess_mode`:
        the ControlNets' residuals carry diffusers' guess-mode scales and, with CFG, see only the conditional half
        (latents, the second half of `side_prompt_embeds`, `control_image` of batch B).
        coef [n,8] from `DDIMScheduler.step_coefficients`; `noise_fn(i)` supplies
        the eta > 0 variance noise of step i; `ucoef` [n,12] (`UniPCMultistepScheduler.unipc_coefficients`) selects
        the UniPC step kernel instead of DDIM; `blend` = dict(x0 [1,4,h,w], mask [1,1,h,w], noise [B,4,h,w],
        sqrt_alpha [n]) is the 4-channel-UNet blend (ref pipeline_PowerPaint.py:1025-1035).
        `callback(i, t, latents_nchw)` may return replacement
        latents. Returns the final latents [B,4,h,w] fp32."""
        B, _, h, w = latents.shape
        nb = prompt_embeds.shape[0]
        do_cfg = nb == 2 * B
        if not do_cfg and nb != B:
            raise ValueError("prompt_embeds batch must be B or 2B")
        n_steps = len(timesteps)
        if n_steps > MAX_STEPS:
            raise ValueError(f"at most {MAX_STEPS} steps")
        extra_per_copy = extra is not None and do_cfg and extra.shape[0] == nb
        if extra is not None and extra.shape[0] not in (B, nb):
            raise ValueError("extra batch must be B or 2B")
        dev = self.unet.device
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)
        multi = isinstance(control_image, (list, tuple))
        if multi:
            n_side = len(control_image)
            if self.mode != "controlnet" or not 1 <= n_side <= len(self._side_nets()):
                raise ValueError(f"{n_side} control images for {len(self._side_nets())} ControlNets")
            scales = [float(v) for v in side_scale]
            keeps = side_keep if side_keep is not None else [None] * n_side
            if len(scales) != n_side or len(keeps) != n_side:
                raise ValueError("control_image, side_scale and side_keep need one entry per ControlNet")
        else:
            n_side, scales, keeps = 1, [float(side_scale)], [side_keep]
        if guess_mode and self.mode != "controlnet":
            raise ValueError("guess_mode applies to ControlNets")
        for kp in keeps:
            if kp is not None and len(kp) != n_steps:
                raise ValueError("side_keep needs one entry per step")
        cur = torch.cuda.current_stream(dev)
        self._stream.wait_stream(cur)
        with torch.cuda.device(dev), torch.cuda.stream(self._stream):
            sched = "unipc" if ucoef is not None else "ddim"
            if sched == "unipc" and (noise_fn is not None or blend is not None):
                raise NotImplementedError("eta / the 4-channel blend are DDIM-only on the fused path")
            st = self._get(B, h, w, do_cfg, prompt_embeds.shape[1], noise_fn is not None, extra_per_copy, sched,
                           blend is not None, n_side if self.side is not None else 0, bool(guess_mode))
            if sched == "unipc":
                if len(ucoef) != n_steps:
                    raise ValueError("ucoef needs one row per step")
                st["ucoef"][:n_steps].copy_(ucoef.to(dev, torch.float32))
                for k in ("last_sample", "m1", "m2"):
                    st[k].zero_()
            # ---- per-call inputs (all outside the loop)
            st["latents"].copy_(ops.nhwc_fp32_from_nchw(latents.to(dev)))
            if extra is not None:
                st["extra"].copy_(ops.nhwc_fp32_from_nchw(extra.to(dev)))
            else:
                st["extra"].zero_()
            self._fill_x_in(st)
            ts = torch.as_tensor([float(t) for t in timesteps], dtype=torch.float32)
            st["timesteps"][:n_steps].copy_(ts.to(dev))
            cf = coef.clone().float()
            cf[:, COEF_GUIDANCE] = float(guidance_scale)
            ss = torch.empty(n_steps, max(n_side, 1))
            for k, (scale, kp) in enumerate(zip(scales, keeps)):
                keep = torch.ones(n_steps) if kp is None else torch.tensor([float(v) for v in kp])
                ss[:, k] = scale * keep
            if blend is not None:
                cf[:, 7] = torch.as_tensor(blend["sqrt_alpha"], dtype=torch.float32)
                st["blend_x0"].copy_(ops.nhwc_fp32_from_nchw(blend["x0"][:1].to(dev))[0])
                st["blend_mask"].copy_(blend["mask"][:1].to(dev, torch.float32).reshape(-1))
                st["blend_noise"].copy_(ops.nhwc_fp32_from_nchw(blend["noise"].to(dev)))
            st["coef"][:n_steps].copy_(cf.to(dev))
            st["side_scale"][:n_steps].copy_(ss.to(dev))
            st["step_idx"].zero_()
            st["uplan"].inputs["ctx"].copy_(prompt_embeds.to(dev, torch.bfloat16))
            if st["side_plans"]:
                if side_prompt_embeds is None:
                    raise ValueError("side_prompt_embeds required")
                if guess_mode and do_cfg:
                    side_prompt_embeds = side_prompt_embeds[B:]  # prompt_embeds.chunk(2)[1] (:1672-1676)
                images = list(control_image) if multi else [control_image]
                for k, sp in enumerate(st["side_plans"]):
                    sp.inputs["ctx"].copy_(side_prompt_embeds.to(dev, torch.bfloat16))
                    if self.mode == "controlnet":
                        if images[k] is None:
                            raise ValueError("control_image required")
                        ci = sp.inputs["cond_in"]
                        ci.copy_(ops.nchw_to_nhwc(images[k].to(dev).float().contiguous(), ci.shape[-1]).view_as(ci))
                        sp.cond_program.run()
            st["ctx_program"].run()
            # ---- the loop
            prog = st["program"]
            if use_graph and callback is None and noise_fn is None:
                if not st["graph"]:
                    prog.build_graph()  # capture does not execute: device state is untouched
                    st["graph"] = True
                for _ in range(n_steps):
                    prog.launch()
            else:
                for i in range(n_steps):
                    if noise_fn is not None:
                        st["noise"].copy_(ops.nhwc_fp32_from_nchw(noise_fn(i).to(dev)))
                    prog.run()
                    if callback is not None:
                        cur_lat = ops.nchw_from_nhwc_fp32(st["latents"], h, w)
                        new = callback(i, timesteps[i], cur_lat)
                        if new is not None and new is not cur_lat:
                            st["latents"].copy_(ops.nhwc_fp32_from_nchw(new.to(dev)))
                            self._fill_x_in(st, latents_only=True)
            out = ops.nchw_from_nhwc_fp32(st["latents"], h, w).clone()
        cur.wait_stream(self._stream)
        out.record_stream(cur)
        return out
