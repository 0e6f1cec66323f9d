"""Host-side planner of the per-step UNet / BrushNet / ControlNet forward.

`NetEngine` takes a diffusers-named state dict (SURVEY.md App. B) for one of the three nets
of the hot path, repacks the weights once (bf16, K-major, conv taps unrolled along K, GEGLU
rows tile-interleaved, all `time_emb_proj` layers stacked into one matrix), and for a given
(batch, h, w) records the whole forward as a `pp_program` of CUDA launches over static
channels-last bf16 buffers:

  reference dataflow                               here
  ------------------------------------------------ ---------------------------------------------
  GroupNorm -> SiLU -> Conv2d (ResnetBlock2D)      pp_group_norm (also does the skip concat)
                                                   -> implicit-GEMM conv with bias + time-embedding
                                                   row + shortcut + BrushNet add in the epilogue
  NCHW<->token permutes (Transformer2DModel)       none: NHWC *is* the token layout
  to_q/to_k/to_v, SDPA, to_out + residual          QK GEMM + V^T GEMM -> pp_attention -> GEMM(+res)
  cross-attn K/V of the prompt, every step         projected once per prompt (`set_context`)
  GEGLU proj, chunk, gelu, mul, Linear + residual  one GEMM with the gate in the epilogue + GEMM(+res)
  22 x time_emb_proj(silu(emb))                    one stacked GEMM per step
  BrushNet 28 zero-convs * scale, 28 adds in UNet  1x1 GEMMs with alpha; adds ride the producer's
                                                   epilogue as the second residual

Reference anchors: powerpaint/models/unet_2d_condition.py:1040-1363 (UNet forward and BrushNet /
ControlNet hooks), powerpaint/models/unet_2d_blocks.py:756,1237,1405,2458,2646 (blocks),
powerpaint/models/BrushNet_CA.py:690-952 (BrushNet forward), SURVEY.md App. A (diffusers blocks).
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from . import _native as N
from . import ops

BF16 = torch.bfloat16


def _ceil(a: int, b: int) -> int:
    return (a + b - 1) // b * b


@dataclass
class NetConfig:
    """The diffusers config keys the hot path reads."""
    in_channels: int = 9
    out_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280)
    layers_per_block: int = 2
    attention_head_dim: int = 8  # number of heads (diffusers naming quirk)
    cross_attention_dim: int = 768
    norm_num_groups: int = 32
    norm_eps: float = 1e-5
    down_block_types: Tuple[str, ...] = ("CrossAttnDownBlock2D", "CrossAttnDownBlock2D",
                                         "CrossAttnDownBlock2D", "DownBlock2D")
    up_block_types: Tuple[str, ...] = ("UpBlock2D", "CrossAttnUpBlock2D", "CrossAttnUpBlock2D",
                                       "CrossAttnUpBlock2D")
    mid_block_scale_factor: float = 1.0
    conditioning_channels: int = 5       # BrushNet
    controlnet_cond_channels: int = 3    # ControlNet
    conditioning_embedding_out_channels: Tuple[int, ...] = (16, 32, 96, 256)


class Plan:
    """A recorded forward for fixed (batch, h, w): programs + the static buffers they touch."""

    def __init__(self):
        self.program: Optional[ops.Program] = None       # per-step forward
        self.ctx_program: Optional[ops.Program] = None   # per-prompt cross-attention K / V^T
        self.cond_program: Optional[ops.Program] = None  # ControlNet: per-control-image embedding
        self.inputs: Dict[str, torch.Tensor] = {}
        self.outputs: Dict[str, object] = {}
        self.bytes = 0                         # bytes of distinct activation storage (after reuse)
        self.buffers: List[torch.Tensor] = []  # every raw activation block (uint8), in allocation order
        self.gn_arenas: Dict[int, list] = {}   # per program: [GroupNorm scratch arena, floats used]
        self.free: Dict[int, List[torch.Tensor]] = {}  # size -> raw blocks whose last reader has been recorded
        self.raw_of: Dict[int, torch.Tensor] = {}      # data_ptr of a live view -> its raw block
        self.chan_stats: Dict[int, tuple] = {}         # data_ptr of a tensor -> (partials, geometry) its producer emits
        self.splitk_flags: Optional[torch.Tensor] = None  # split-K hand-over flags shared by the plan's launches (kept at zero)
        self.row_stats: Dict[int, torch.Tensor] = {}   # data_ptr of a tensor -> per-row {rstd, -rstd mean} its producer leaves
        self.row_ticket: Optional[torch.Tensor] = None  # arrival counters of the LayerNorm-statistics producers (kept at zero)
        self.scale_dev: Optional[torch.Tensor] = None  # eager side-net forward: 1-float conditioning scale


class NetEngine:
    KINDS = ("unet", "brushnet", "controlnet")
    GN_ARENA_BYTES = 32 << 20  # GroupNorm scratch per program (SD-1.5 UNet: 61 layers x <= 320 KB); grows on demand
    # GroupNorm statistics from the producing GEMM's epilogue (PP_B200_GN_FUSED=0: standalone statistics pass)
    GN_FUSED = os.environ.get("PP_B200_GN_FUSED", "1") != "0"

    def __init__(self, cfg: NetConfig, state_dict: Dict[str, torch.Tensor], kind: str = "unet",
                 device: Optional[torch.device] = None):
        if kind not in self.KINDS:
            raise ValueError(f"kind must be one of {self.KINDS}")
        self.cfg = cfg
        self.kind = kind
        self.device = torch.device(device or "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("NetEngine needs a CUDA device: the hot path has no CPU fallback")
        N.lib()  # fail loudly if the extension is missing
        self._sd = state_dict
        self._w: Dict[str, torch.Tensor] = {}
        self._plans: Dict[tuple, Plan] = {}
        for t in cfg.down_block_types:
            if t not in ("CrossAttnDownBlock2D", "DownBlock2D"):
                raise NotImplementedError(f"down block type {t} is outside the SD-1.5 hot path")
        for t in cfg.up_block_types:
            if t not in ("CrossAttnUpBlock2D", "UpBlock2D"):
                raise NotImplementedError(f"up block type {t} is outside the SD-1.5 hot path")
        if cfg.block_out_channels[0] % 8 or any(c % 8 for c in cfg.block_out_channels):
            raise ValueError("block_out_channels must be multiples of 8")
        self._pack_time_proj()

    # ------------------------------------------------------------------ weights
    def _raw(self, name: str) -> torch.Tensor:
        if name not in self._sd:
            raise KeyError(f"missing weight '{name}' in state dict")
        return self._sd[name].detach().to(self.device, torch.float32)

    def _cached(self, key: str, fn):
        t = self._w.get(key)
        if t is None:
            t = fn()
            self._w[key] = t
        return t

    def w_linear(self, name: str) -> torch.Tensor:
        return self._cached("lin:" + name, lambda: ops.pack_linear_weight(self._raw(name + ".weight")))

    def w_conv3(self, name: str, split: Optional[int] = None, pad_in: Optional[int] = None) -> torch.Tensor:
        def make():
            w = self._raw(name + ".weight")
            if pad_in is not None and pad_in > w.shape[1]:
                wp = torch.zeros(w.shape[0], pad_in, 3, 3, device=w.device)
                wp[:, : w.shape[1]] = w
                w = wp
            return ops.pack_conv3x3_weight(w, split)
        return self._cached(f"c3:{name}:{split}:{pad_in}", make)

    def w_concat_linear(self, name: str, split: int) -> torch.Tensor:
        return self._cached(f"cl:{name}:{split}",
                            lambda: ops.pack_concat_linear_weight(self._raw(name + ".weight"), split))

    def w_qk(self, prefix: str) -> torch.Tensor:
        return self._cached("qk:" + prefix, lambda: torch.cat(
            [self._raw(prefix + ".to_q.weight"), self._raw(prefix + ".to_k.weight")], 0).to(BF16).contiguous())

    # LayerNorm folded into the GEMMs either side of it (PP_B200_LN_FOLD=0: standalone LayerNorm kernel)
    LN_FOLD = os.environ.get("PP_B200_LN_FOLD", "1") != "0"
    # to_q | to_k | to_v^T of a self-attention as one launch (PP_B200_QKV_MERGED=0: q|k and V^T separately)
    QKV_MERGED = os.environ.get("PP_B200_QKV_MERGED", "1") != "0"

    def w_ln_folded(self, key: str, wnames, ln_name: str, bias_name: Optional[str] = None, geglu: bool = False):
        """Weights of the GEMM that consumes LayerNorm(x): y = LN(x) W^T + b = rstd (x W'^T - mean u) + b' with
        W' = W * gamma (bf16), u = row sums of the bf16 W' (what the tensor core multiplies), b' = W beta + b.
        Returns (W' bf16 [N, K], u fp32 [N], b' fp32 [N]); `geglu`: rows tile-interleaved like `w_geglu`."""
        def make():
            w = torch.cat([self._raw(n + ".weight").reshape(self._raw(n + ".weight").shape[0], -1) for n in wnames], 0)
            wf, u, b = ops.fold_layer_norm_into_linear(w, self._raw(ln_name + ".weight"), self._raw(ln_name + ".bias"),
                                                       self._raw(bias_name) if bias_name is not None else None)
            if geglu:  # value / gate rows interleaved per tile; u and b' ride the same permutation
                wi, u = ops.pack_geglu_weight(wf.float(), u, self.GEGLU_BLOCK_N)
                _, b = ops.pack_geglu_weight(wf.float(), b, self.GEGLU_BLOCK_N)
                wf = wi  # bf16 -> fp32 -> bf16 is exact
            return wf.contiguous(), u.float().contiguous(), b.float().contiguous()
        return self._cached("lnf:" + key, make)

    # tile width of the GEGLU GEMMs (weights are interleaved per tile; 256: the fixed per-tile cost of the epilogue is paid half
    # as often: 118 -> 108 us at 320 -> 2560, M = 65536). PP_B200_GEGLU_BN=128|256
    GEGLU_BLOCK_N = int(os.environ.get("PP_B200_GEGLU_BN", "256"))

    def w_geglu(self, name: str):
        def make():
            return ops.pack_geglu_weight(self._raw(name + ".weight"), self._raw(name + ".bias"), self.GEGLU_BLOCK_N)
        return self._cached("gg:" + name, make)

    def vec(self, name: str) -> torch.Tensor:
        return self._cached("v:" + name, lambda: self._raw(name).contiguous())

    def _resnet_names(self) -> List[str]:
        cfg = self.cfg
        names = []
        for i in range(len(cfg.down_block_types)):
            for j in range(cfg.layers_per_block):
                names.append(f"down_blocks.{i}.resnets.{j}")
        names += ["mid_block.resnets.0", "mid_block.resnets.1"]
        if self.kind != "controlnet":
            for i in range(len(cfg.up_block_types)):
                for j in range(cfg.layers_per_block + 1):
                    names.append(f"up_blocks.{i}.resnets.{j}")
        return names

    def _pack_time_proj(self):
        """stack every resnet's time_emb_proj into one [sum(Cout), 4*C0] matrix"""
        ws, bs, self._tp_off = [], [], {}
        off = 0
        for n in self._resnet_names():
            w = self._raw(n + ".time_emb_proj.weight")
            self._tp_off[n] = (off, w.shape[0])
            off += w.shape[0]
            ws.append(w)
            bs.append(self._raw(n + ".time_emb_proj.bias"))
        self._tp_total = off
        self._w["tp:w"] = torch.cat(ws, 0).to(BF16).contiguous()
        self._w["tp:b"] = torch.cat(bs, 0).contiguous()

    # ------------------------------------------------------------------ planning helpers
    def _buf(self, plan: Plan, *shape, dtype=BF16) -> torch.Tensor:
        """An activation buffer of the plan. Storage is recycled: a block whose last reader has been
        recorded (`_free`) serves later buffers of the same size — ops run in stream order (also inside
        the captured graph), so a later writer can never overtake an earlier reader."""
        numel = 1
        for d in shape:
            numel *= int(d)
        item = torch.empty(0, dtype=dtype).element_size()
        nbytes = (numel * item + 255) // 256 * 256
        pool = plan.free.get(nbytes)
        if pool:
            raw = pool.pop()
        else:
            raw = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            plan.bytes += nbytes
            plan.buffers.append(raw)
        t = raw.view(dtype)[:numel].view(*shape)
        plan.raw_of[t.data_ptr()] = raw
        return t

    def _free(self, plan: Plan, *tensors) -> None:
        """every op reading or writing these buffers has been recorded: their storage may be reused"""
        for t in tensors:
            if t is None:
                continue
            raw = plan.raw_of.pop(t.data_ptr(), None)
            if raw is None:
                continue  # not a plan buffer (a weight, a shared input) or already released
            ent = plan.chan_stats.pop(t.data_ptr(), None)
            rec = plan.row_stats.pop(t.data_ptr(), None)
            plan.free.setdefault(raw.numel(), []).append(raw)
            if ent is not None:
                self._free(plan, ent[0])  # the producer's partial sums die with the tensor they describe
            if rec is not None:
                self._free(plan, rec)

    # split-K x2 for long-K launches whose tiles fill at most half of the GPU. Off by default: measured neutral (8x8 conv
    # 1280 -> 1280: 40.9 us plain, 40.6 us split) — those layers are bound by L2 serving the same weight / activation
    # tiles to every CTA, not by the number of busy SMs (profiles/r02_notes.md). PP_B200_SPLITK=1 switches it on.
    SPLITK = os.environ.get("PP_B200_SPLITK", "0") == "1"

    def _with_splitk(self, plan: Plan, desc):
        """hand the launch a split-K workspace if it could use one; returns the scratch to release after recording"""
        if not self.SPLITK:
            return None
        nbytes, tiles = ops.gemm_splitk_query(desc)
        if nbytes <= 0:
            return None
        ws = self._buf(plan, nbytes // 4, dtype=torch.float32)
        if plan.splitk_flags is None or plan.splitk_flags.numel() < tiles:
            plan.splitk_flags = torch.zeros(max(tiles, 4096), dtype=torch.int32, device=self.device)  # self-resetting
            plan.buffers.append(plan.splitk_flags)
        ops.attach_splitk(desc, ws, plan.splitk_flags)
        return ws

    def _with_stats(self, plan: Plan, desc, out: torch.Tensor) -> None:
        """let this GEMM / conv emit the GroupNorm partial sums of its output from the epilogue"""
        if not self.GN_FUSED:
            return
        g = ops.gemm_stats_geometry(desc)
        if not g.supported:
            return
        part = self._buf(plan, int(g.bytes) // 4, dtype=torch.float32)
        ops.attach_chan_stats(desc, part)
        plan.chan_stats[out.data_ptr()] = (part, g)

    def _gn(self, plan, prog, x0, x1, nb, hw, name, eps, silu):
        c0 = x0.shape[-1]
        c1 = x1.shape[-1] if x1 is not None else 0
        groups = self.cfg.norm_num_groups
        y = self._buf(plan, nb, hw, c0 + c1)
        # the sum / sum-of-squares scratch of every GroupNorm of this plan lives in arenas that a single
        # memset at the head of the program clears (one graph node per step instead of one per GroupNorm)
        key = id(prog)
        need = (ops.gn_scratch_bytes(nb, hw, c0 + c1, groups) + 255) // 256 * 64  # floats, 256-byte slots
        ent = plan.gn_arenas.get(key)
        if ent is None or ent[1] + need > ent[0].numel():
            arena = torch.zeros(max(self.GN_ARENA_BYTES // 4, need), dtype=torch.float32, device=self.device)
            plan.bytes += arena.numel() * 4
            plan.buffers.append(arena)
            prog.add_memset(arena)
            ent = plan.gn_arenas[key] = [arena, 0]
        arena, used = ent
        stats = arena[used:used + need]
        ent[1] = used + need
        s0 = plan.chan_stats.get(x0.data_ptr())
        s1 = plan.chan_stats.get(x1.data_ptr()) if x1 is not None else None
        fused = s0 is not None and (x1 is None or s1 is not None)
        prog.add(ops.gn_desc(x0=x0, x1=x1, c0=c0, c1=c1, batch=nb, hw=hw, groups=groups,
                             gamma=self.vec(name + ".weight"), beta=self.vec(name + ".bias"), eps=eps, silu=silu,
                             stats=stats, y=y, stats_prezeroed=True,
                             part0=s0[0] if fused else None, geom0=s0[1] if fused else None,
                             part1=s1[0] if fused and s1 is not None else None,
                             geom1=s1[1] if fused and s1 is not None else None))
        return y

    def _conv3(self, plan, prog, x, nb, h, w, name, cout, *, stride2=False, rowvec=None, res1=None, res2=None,
               alpha=1.0, out_fp32=False, pad_in=None, out=None, stats=False, act=N.PP_ACT_NONE, a_mode=None,
               ldc=0):
        cin = x.shape[-1]
        if a_mode is None:
            a_mode = N.PP_A_CONV3X3_S2 if stride2 else N.PP_A_CONV3X3
        if a_mode == N.PP_A_CONV3X3_S2:
            ho, wo = (h + 1) // 2, (w + 1) // 2
        elif a_mode == N.PP_A_CONV3X3_S2P0:
            ho, wo = h // 2, w // 2
        else:
            ho, wo = h, w
        if out is None:
            out = self._buf(plan, nb, ho * wo, cout, dtype=torch.float32 if out_fp32 else BF16)
        rv, rv_ld = (None, 0) if rowvec is None else rowvec
        desc = ops.gemm_desc(a0=x, w=self.w_conv3(name, pad_in=pad_in), out=out, N_=cout, a_mode=a_mode, c0=cin,
                             nb=nb, h=h, w_=w, bias=self.vec(name + ".bias"), rowvec=rv, rowvec_ld=rv_ld, res1=res1,
                             res2=res2, alpha=alpha, out_fp32=out_fp32, act=act, ldc=ldc)
        if stats:
            self._with_stats(plan, desc, out)
        ws = self._with_splitk(plan, desc)
        prog.add(desc)
        self._free(plan, ws)  # scratch of this one launch
        return out

    def _linear(self, plan, prog, x, M, wname, n_out, *, w=None, bias=None, res1=None, res2=None, alpha=1.0,
                act=N.PP_ACT_NONE, out=None, out_fp32=False, a1=None, c1=0, ldc=0, lda0=0, stats_hw=0,
                alpha_dev=None, alpha_step=None, alpha_stride=0, row_stats=False, ln=None):
        """`stats_hw` > 0: rows per sample; the GEMM then emits GroupNorm partial sums of its output.
        `row_stats`: also emit the per-row LayerNorm records of the output (returned as `plan.row_stats[out]`);
        `ln` = (records, u, eps): LayerNorm of `x` folded into this GEMM."""
        if out is None:
            out = self._buf(plan, M, n_out, dtype=torch.float32 if out_fp32 else BF16)
        desc = ops.gemm_desc(a0=x, a1=a1, c1=c1, w=w if w is not None else self.w_linear(wname), out=out, N_=n_out,
                             M=M, bias=bias, res1=res1, res2=res2, alpha=alpha, act=act, out_fp32=out_fp32,
                             ldc=ldc, lda0=lda0, rows_per_group=stats_hw, alpha_dev=alpha_dev,
                             alpha_step=alpha_step, alpha_stride=alpha_stride, ln=ln)
        if stats_hw:
            self._with_stats(plan, desc, out)
        rec = None
        if row_stats:
            nrec = ops.gemm_row_stats_records(desc)
            if nrec > 0:
                # per-row LayerNorm statistics of the output: the records are scratch of this one launch (the CTA
                # finishing a row block folds them into `final`), the ticket array is shared by all producers of the plan
                rec = self._buf(plan, nrec, M, 4, dtype=torch.float32)
                final = self._buf(plan, M, 2, dtype=torch.float32)
                n_t = _ceil(M, 128) // 128
                if plan.row_ticket is None or plan.row_ticket.numel() < n_t:
                    plan.row_ticket = torch.zeros(max(n_t, 1024), dtype=torch.int32, device=self.device)
                    plan.buffers.append(plan.row_ticket)
                ops.attach_row_stats(desc, rec, final, plan.row_ticket, 1e-5)
                plan.row_stats[out.data_ptr()] = final
        prog.add(desc)
        if rec is not None:
            self._free(plan, rec)
        return out

    def _ln_of(self, plan, x):
        """per-row LayerNorm records of x emitted by its producer, or None (then the standalone kernel runs)"""
        return plan.row_stats.get(x.data_ptr()) if self.LN_FOLD else None

    def _resnet(self, plan, prog, name, x0, x1, nb, h, w, cout, tproj, *, out_scale=1.0, add=None):
        """ResnetBlock2D on the (virtual) concat of x0 and x1 (SURVEY.md App. A.1)."""
        hw = h * w
        c0 = x0.shape[-1]
        c1 = x1.shape[-1] if x1 is not None else 0
        cin = c0 + c1
        eps = self.cfg.norm_eps
        n1 = self._gn(plan, prog, x0, x1, nb, hw, name + ".norm1", eps, True)
        off, tc = self._tp_off[name]
        assert tc == cout
        t1 = self._conv3(plan, prog, n1, nb, h, w, name + ".conv1", cout,
                         rowvec=(tproj[:, off:off + cout], self._tp_total), stats=True)
        self._free(plan, n1)
        n2 = self._gn(plan, prog, t1, None, nb, hw, name + ".norm2", eps, True)
        self._free(plan, t1)
        sc_owned = None
        if cin != cout or x1 is not None:
            # 1x1 conv_shortcut over the concat: two A sources walked along K
            if (name + ".conv_shortcut.weight") not in self._sd:
                raise KeyError(f"{name}: in != out channels but no conv_shortcut weight")
            if x1 is not None:
                wsc = self.w_concat_linear(name + ".conv_shortcut", c0)
                sc = self._buf(plan, nb * hw, cout)
                prog.add(ops.gemm_desc(a0=x0, a1=x1, c0=c0, c1=c1, w=wsc, out=sc, N_=cout, M=nb * hw,
                                       bias=self.vec(name + ".conv_shortcut.bias")))
            else:
                sc = self._linear(plan, prog, x0, nb * hw, name + ".conv_shortcut", cout,
                                  bias=self.vec(name + ".conv_shortcut.bias"))
            sc_owned = sc
        else:
            sc = x0
        out = self._conv3(plan, prog, n2, nb, h, w, name + ".conv2", cout, res1=sc, res2=add, alpha=1.0 / out_scale,
                          stats=True)
        self._free(plan, n2, sc_owned)
        return out

    def _transformer(self, plan, ctxprog, prog, name, x, nb, h, w, heads, ctx, *, add=None):
        """Transformer2DModel with one BasicTransformerBlock (SURVEY.md App. A.2-A.5)."""
        hw = h * w
        M = nb * hw
        C = x.shape[-1]
        d = C // heads
        scale = 1.0 / math.sqrt(d)
        g = self._gn(plan, prog, x, None, nb, hw, name + ".norm", 1e-6, False)
        fold = self.LN_FOLD
        t0 = self._linear(plan, prog, g, M, name + ".proj_in", C, bias=self.vec(name + ".proj_in.bias"), row_stats=fold)
        self._free(plan, g)
        b = name + ".transformer_blocks.0"
        hw_ld = _ceil(hw, 8)
        # --- self attention. LayerNorm (norm1) is folded into q|k and V^T: the producer of t0 left per-row records,
        # the consumers multiply the raw t0 by W * gamma and finish the normalisation in their epilogues
        rec = self._ln_of(plan, t0)
        vt = self._buf(plan, nb, C, hw_ld, dtype=torch.float16)  # fp16 V^T: P is fp16 in pp_attention
        # to_q | to_k | to_v^T in ONE launch when the tiles line up (whole 128-token tiles per sample, the V columns
        # start on a tile boundary): t0 is read once, the V tiles leave through a transposed staging tile
        qkv_bn = 160 if C % 160 == 0 else 128 if C % 128 == 0 else 0
        merged = self.QKV_MERGED and qkv_bn and hw % 128 == 0
        if merged:
            names = [b + ".attn1.to_q", b + ".attn1.to_k", b + ".attn1.to_v"]
            if rec is not None:
                wqkv, uqkv, bqkv = self.w_ln_folded(b + ".attn1.qkv", names, b + ".norm1")
                a_in, ln1 = t0, (rec, uqkv, 1e-5)
            else:
                l1 = self._buf(plan, M, C)
                prog.add_layer_norm(t0, l1, self.vec(b + ".norm1.weight"), self.vec(b + ".norm1.bias"), M, C, 1e-5)
                wqkv = self._cached("qkv:" + b, lambda: torch.cat([self._raw(n + ".weight") for n in names], 0)
                                    .to(BF16).contiguous())
                bqkv, a_in, ln1 = None, l1, None
            qk = self._buf(plan, M, 2 * C)
            prog.add(ops.gemm_desc(a0=a_in, w=wqkv, out=qk, N_=3 * C, M=M, bias=bqkv, ln=ln1, block_n=qkv_bn,
                                   epilogue=N.PP_EPI_ROWS_THEN_TRANSPOSED, out_t=vt, trans_from_col=2 * C, t_rows=hw,
                                   t_ld=hw_ld, t_fp16=True))
            if rec is None:
                self._free(plan, a_in)
        elif rec is not None:
            wqk, uqk, bqk = self.w_ln_folded(b + ".attn1.qk", [b + ".attn1.to_q", b + ".attn1.to_k"], b + ".norm1")
            wv, uv, bv = self.w_ln_folded(b + ".attn1.v", [b + ".attn1.to_v"], b + ".norm1")
            qk = self._linear(plan, prog, t0, M, None, 2 * C, w=wqk, bias=bqk, ln=(rec, uqk, 1e-5))
            prog.add(ops.gemm_desc(a0=t0, w=wv, out=vt, N_=C, M=M, bias=bv, epilogue=N.PP_EPI_TRANSPOSED, t_rows=hw,
                                   t_ld=hw_ld, t_fp16=True, ln=(rec, uv, 1e-5)))
        else:
            l1 = self._buf(plan, M, C)
            prog.add_layer_norm(t0, l1, self.vec(b + ".norm1.weight"), self.vec(b + ".norm1.bias"), M, C, 1e-5)
            qk = self._linear(plan, prog, l1, M, None, 2 * C, w=self.w_qk(b + ".attn1"))
            prog.add(ops.gemm_desc(a0=l1, w=self.w_linear(b + ".attn1.to_v"), out=vt, N_=C, M=M,
                                   epilogue=N.PP_EPI_TRANSPOSED, t_rows=hw, t_ld=hw_ld, t_fp16=True))
            self._free(plan, l1)
        a1 = self._buf(plan, M, C)
        prog.add(ops.attn_desc(q=qk, k=qk[:, C:], vt=vt, out=a1, batch=nb, heads=heads, d=d, nq=hw, nk=hw,
                               q_ld=2 * C, k_ld=2 * C, vt_ld=hw_ld, o_ld=C, q_batch_stride=hw * 2 * C,
                               k_batch_stride=hw * 2 * C, scale=scale))
        self._free(plan, qk, vt)
        t1 = self._linear(plan, prog, a1, M, b + ".attn1.to_out.0", C, bias=self.vec(b + ".attn1.to_out.0.bias"), res1=t0,
                          row_stats=fold)
        self._free(plan, a1, t0)
        # --- cross attention (K / V^T of the prompt are projected once per prompt: never recycled)
        rec = self._ln_of(plan, t1)
        if rec is not None:
            wq, uq, bq = self.w_ln_folded(b + ".attn2.q", [b + ".attn2.to_q"], b + ".norm2")
            q2 = self._linear(plan, prog, t1, M, None, C, w=wq, bias=bq, ln=(rec, uq, 1e-5))
        else:
            l2 = self._buf(plan, M, C)
            prog.add_layer_norm(t1, l2, self.vec(b + ".norm2.weight"), self.vec(b + ".norm2.bias"), M, C, 1e-5)
            q2 = self._linear(plan, prog, l2, M, b + ".attn2.to_q", C)
            self._free(plan, l2)
        nk = ctx.shape[1]
        nk_ld = _ceil(nk, 8)
        k2 = torch.empty(nb * nk, C, dtype=BF16, device=self.device)
        # zeros: the pad columns nk..nk_ld are never written (nor read: the tensor map ends at nk), keep them clean
        v2t = torch.zeros(nb, C, nk_ld, dtype=torch.float16, device=self.device)
        plan.bytes += (k2.numel() + v2t.numel()) * 2
        self._linear(plan, ctxprog, ctx, nb * nk, b + ".attn2.to_k", C, out=k2)
        ctxprog.add(ops.gemm_desc(a0=ctx, w=self.w_linear(b + ".attn2.to_v"), out=v2t, N_=C, M=nb * nk,
                                  epilogue=N.PP_EPI_TRANSPOSED, t_rows=nk, t_ld=nk_ld, t_fp16=True))
        a2 = self._buf(plan, M, C)
        prog.add(ops.attn_desc(q=q2, k=k2, vt=v2t, out=a2, batch=nb, heads=heads, d=d, nq=hw, nk=nk, q_ld=C, k_ld=C,
                               vt_ld=nk_ld, o_ld=C, q_batch_stride=hw * C, k_batch_stride=nk * C, scale=scale))
        self._free(plan, q2)
        t2 = self._linear(plan, prog, a2, M, b + ".attn2.to_out.0", C, bias=self.vec(b + ".attn2.to_out.0.bias"), res1=t1,
                          row_stats=fold)
        self._free(plan, a2, t1)
        # --- feed-forward (GEGLU), norm3 folded the same way
        rec = self._ln_of(plan, t2)
        if rec is not None:
            wg, ug, bg = self.w_ln_folded(b + ".ff.geglu", [b + ".ff.net.0.proj"], b + ".norm3",
                                          bias_name=b + ".ff.net.0.proj.bias", geglu=True)
            ln3, a_ff = (rec, ug, 1e-5), t2
        else:
            l3 = self._buf(plan, M, C)
            prog.add_layer_norm(t2, l3, self.vec(b + ".norm3.weight"), self.vec(b + ".norm3.bias"), M, C, 1e-5)
            wg, bg = self.w_geglu(b + ".ff.net.0.proj")
            ln3, a_ff = None, l3
        F_ = wg.shape[0] // 2
        ffh = self._buf(plan, M, F_)
        prog.add(ops.gemm_desc(a0=a_ff, w=wg, out=ffh, N_=2 * F_, M=M, bias=bg, epilogue=N.PP_EPI_GEGLU,
                               block_n=self.GEGLU_BLOCK_N, ln=ln3))
        if ln3 is None:
            self._free(plan, a_ff)
        t3 = self._linear(plan, prog, ffh, M, b + ".ff.net.2", C, bias=self.vec(b + ".ff.net.2.bias"), res1=t2)
        self._free(plan, ffh, t2)
        # --- proj_out + the Transformer2DModel residual (+ BrushNet add)
        out = self._linear(plan, prog, t3, M, name + ".proj_out", C, bias=self.vec(name + ".proj_out.bias"),
                           res1=x, res2=add, stats_hw=hw)
        self._free(plan, t3)
        return out

    # ------------------------------------------------------------------ plan
    MAX_PLANS = 2  # eager-forward plans kept per engine (least recently used is dropped)

    def plan(self, nb: int, h: int, w: int, ctx_len: int = 77, *, with_brushnet_adds: bool = False,
             with_controlnet_res: bool = False, use_step_table: bool = False, n_steps: int = 0,
             brushnet_outputs: bool = False, guess_mode: bool = False) -> Plan:
        key = (nb, h, w, ctx_len, with_brushnet_adds, with_controlnet_res, use_step_table, n_steps, brushnet_outputs,
               guess_mode)
        p = self._plans.pop(key, None)
        if p is None:
            shared = dict(cn_alpha=self.guess_alphas()) if guess_mode else None
            p = self._build_plan(nb, h, w, ctx_len, with_brushnet_adds, with_controlnet_res, use_step_table, n_steps,
                                 shared=shared)
            if self.kind in ("brushnet", "controlnet") and p.scale_dev is None:
                # eager forward: conditioning_scale is read from a device scalar at run time
                p.scale_dev = torch.ones(1, dtype=torch.float32, device=self.device)
            if brushnet_outputs:
                self.append_brushnet_outputs(p, 1.0, scale_dev=(p.scale_dev, None, 0))
            while len(self._plans) >= self.MAX_PLANS:
                self._plans.pop(next(iter(self._plans)))
        self._plans[key] = p  # most recently used last
        return p

    def guess_alphas(self):
        """(down, mid) constant factors of a ControlNet's residuals in guess mode: diffusers' ControlNetModel.forward
        scales the down residuals by torch.logspace(-1, 0, n_down + 1)[:n_down] and the mid residual by its last
        entry (1.0), each times conditioning_scale (which stays the device-side factor)"""
        n_down = len(self._state_shapes(1, 64, 64)[0])
        s = torch.logspace(-1, 0, n_down + 1, dtype=torch.float32).tolist()
        return s[:n_down], s[-1]

    @staticmethod
    def _levels(h: int, w: int, n: int):
        """(h, w) at each of the n resolutions: every Downsample2D (3x3, stride 2, pad 1) maps h -> ceil(h / 2)"""
        out = [(h, w)]
        for _ in range(n - 1):
            h, w = (h + 1) // 2, (w + 1) // 2
            out.append((h, w))
        return out

    def _state_shapes(self, nb, h, w):
        """(channels, h, w) of the 12 down states, the mid state and the 15 up states"""
        cfg = self.cfg
        boc = cfg.block_out_channels
        lv = self._levels(h, w, len(boc))
        down = [(boc[0],) + lv[0]]
        for i, c in enumerate(boc):
            for _ in range(cfg.layers_per_block):
                down.append((c,) + lv[i])
            if i != len(boc) - 1:
                down.append((c,) + lv[i + 1])
        mid = (boc[-1],) + lv[-1]
        up = []
        n = len(boc)
        for i, c in enumerate(reversed(boc)):
            for _ in range(cfg.layers_per_block + 1):
                up.append((c,) + lv[n - 1 - i])
            if i != n - 1:
                up.append((c,) + lv[n - 2 - i])
        return down, mid, up

    def _build_plan(self, nb, h, w, ctx_len, with_adds, with_cn, use_step_table, n_steps,
                    shared: Optional[dict] = None) -> Plan:
        """`shared` lets several nets record into ONE program over common inputs (the fused
        per-step pipeline): keys `program`, `ctx_program`, `x_in` (a [nb, h*w, C] buffer whose
        first channels are this net's input; extra channels meet zero weights), `timesteps`,
        `step_idx`, `plan` (record into an existing Plan so that the nets share one buffer pool), and for the
        UNet `adds` = (down, mid, up) / `cn` = (down, mid) buffers produced by the side net;
        `scale_dev` = (tensor, step_idx, stride): device-side conditioning scale of the side net; for a ControlNet
        `cn_out` / `cn_res2` = (down list, mid): buffers its zero-convs write / add after scaling, and
        `cn_alpha` = (down list, mid): constant per-residual factors (`guess_alphas`)."""
        shared = shared or {}
        cfg = self.cfg
        boc = cfg.block_out_channels
        if h < 1 or w < 1:
            raise ValueError(f"latent size {h}x{w} invalid")
        lv = self._levels(h, w, len(boc))
        if len(boc) > 1 and min(lv[-2]) < 2:
            raise ValueError(f"latent size {h}x{w} is too small for {len(boc) - 1} stride-2 convolutions")
        heads = cfg.attention_head_dim
        plan = Plan()
        prog = shared.get("program") or ops.Program()
        ctxprog = shared.get("ctx_program") or ops.Program()
        plan.program, plan.ctx_program = prog, ctxprog
        pool = shared.get("pool")
        if pool is not None:  # the nets of one fused step share one activation pool
            plan.free, plan.raw_of, plan.gn_arenas = pool.free, pool.raw_of, pool.gn_arenas
        C0 = boc[0]
        temb_c = 4 * C0

        def persistent(*shape, dtype=BF16, zero=False):
            t = (torch.zeros if zero else torch.empty)(*shape, dtype=dtype, device=self.device)
            plan.bytes += t.numel() * t.element_size()
            return t

        # ---------------- inputs
        if self.kind == "brushnet":
            cin = cfg.in_channels + cfg.conditioning_channels
            conv_in_name = "conv_in_condition"
        else:
            cin = cfg.in_channels
            conv_in_name = "conv_in"
        if shared.get("x_in") is not None:
            x_in = shared["x_in"]
            cin_pad = x_in.shape[-1]
            if cin_pad < cin or tuple(x_in.shape[:2]) != (nb, h * w):
                raise ValueError("shared x_in has the wrong shape")
        else:
            cin_pad = _ceil(cin, 8)
            x_in = persistent(nb, h * w, cin_pad, zero=True)
        ctx = persistent(nb, ctx_len, cfg.cross_attention_dim, zero=True)
        plan.inputs["x_in"] = x_in
        plan.inputs["ctx"] = ctx
        if shared.get("timesteps") is not None:
            plan.inputs["timesteps"] = shared["timesteps"]
            plan.inputs["step_idx"] = shared["step_idx"]
        elif use_step_table:
            plan.inputs["timesteps"] = torch.zeros(max(n_steps, 1), dtype=torch.float32, device=self.device)
            plan.inputs["step_idx"] = torch.zeros(1, dtype=torch.int32, device=self.device)
        else:
            plan.inputs["timesteps"] = torch.zeros(nb, dtype=torch.float32, device=self.device)
        down_shapes, mid_shape, up_shapes = self._state_shapes(nb, h, w)
        adds_down = adds_up = None
        add_mid = None
        if with_adds:
            if shared.get("adds") is not None:
                adds_down, add_mid, adds_up = shared["adds"]
            else:
                adds_down = [persistent(nb, hh * ww, c, zero=True) for (c, hh, ww) in down_shapes]
                add_mid = persistent(nb, mid_shape[1] * mid_shape[2], mid_shape[0], zero=True)
                adds_up = [persistent(nb, hh * ww, c, zero=True) for (c, hh, ww) in up_shapes]
            plan.inputs["adds_down"], plan.inputs["add_mid"], plan.inputs["adds_up"] = adds_down, add_mid, adds_up
        cn_down = cn_mid = None
        if with_cn:
            if shared.get("cn") is not None:
                cn_down, cn_mid = shared["cn"]
            else:
                cn_down = [persistent(nb, hh * ww, c, zero=True) for (c, hh, ww) in down_shapes]
                cn_mid = persistent(nb, mid_shape[1] * mid_shape[2], mid_shape[0], zero=True)
            plan.inputs["cn_down"], plan.inputs["cn_mid"] = cn_down, cn_mid

        # ---------------- time embedding (unet_2d_condition.py:1155-1156) + stacked time_emb_proj
        tsin = self._buf(plan, nb, C0)
        prog.add_time_embed(plan.inputs["timesteps"], plan.inputs.get("step_idx"), tsin, nb, C0)
        e1 = self._linear(plan, prog, tsin, nb, "time_embedding.linear_1", temb_c,
                          bias=self.vec("time_embedding.linear_1.bias"), act=N.PP_ACT_SILU)
        # resnets consume silu(emb); emb itself is not used elsewhere on the SD-1.5 path
        e2 = self._linear(plan, prog, e1, nb, "time_embedding.linear_2", temb_c,
                          bias=self.vec("time_embedding.linear_2.bias"), act=N.PP_ACT_SILU)
        tproj = self._buf(plan, nb, self._tp_total, dtype=torch.float32)  # read by every resnet: never freed
        prog.add(ops.gemm_desc(a0=e2, w=self._w["tp:w"], out=tproj, N_=self._tp_total, M=nb, bias=self._w["tp:b"],
                               out_fp32=True))
        self._free(plan, tsin, e1, e2)

        # ---------------- conv_in
        hcur = self._conv3(plan, prog, x_in.view(nb, h * w, cin_pad), nb, h, w, conv_in_name, C0, pad_in=cin_pad,
                           stats=True)
        if self.kind == "controlnet":
            cond_in = persistent(nb, (8 * h) * (8 * w), _ceil(cfg.controlnet_cond_channels, 8), zero=True)
            plan.inputs["cond_in"] = cond_in
            cond_emb = persistent(nb, h * w, C0)
            plan.outputs["cond_emb"] = cond_emb
            plan.cond_program = self._build_cond_embedding(plan, cond_in, cond_emb, nb, 8 * h, 8 * w)
            h_sum = self._buf(plan, nb, h * w, C0)
            prog.add_add(hcur, cond_emb, h_sum, hcur.numel())
            self._free(plan, hcur)
            hcur = h_sum
        skips = [(hcur, h, w)]  # pre-add (unet_2d_condition.py:1220 before :1223)
        states_down = [hcur]
        ai = 0
        if with_adds:
            hsum = self._buf(plan, nb, h * w, C0)
            prog.add_add(hcur, adds_down[0], hsum, hcur.numel())
            hcur = hsum
            ai = 1
        # buffers that are only an intermediate `h` (not a skip / captured state) die with their last reader
        transient = [hcur] if with_adds else []

        def next_add(lst, idx):
            return lst[idx] if lst is not None else None

        def retire(t):
            if any(t is u for u in transient):
                self._free(plan, t)

        # ---------------- down
        ch, cw = h, w
        for i, btype in enumerate(cfg.down_block_types):
            cout = boc[i]
            for j in range(cfg.layers_per_block):
                rn = f"down_blocks.{i}.resnets.{j}"
                has_attn = btype == "CrossAttnDownBlock2D"
                add = next_add(adds_down, ai) if with_adds else None
                prev = hcur
                hcur = self._resnet(plan, prog, rn, hcur, None, nb, ch, cw, cout, tproj,
                                    add=None if has_attn else add)
                retire(prev)
                if has_attn:
                    r_out = hcur
                    hcur = self._transformer(plan, ctxprog, prog, f"down_blocks.{i}.attentions.{j}", hcur, nb, ch, cw,
                                             heads, ctx, add=add)
                    self._free(plan, r_out)
                ai += 1 if with_adds else 0
                skips.append((hcur, ch, cw))
                states_down.append(hcur)
            if i != len(boc) - 1:
                add = next_add(adds_down, ai) if with_adds else None
                hcur = self._conv3(plan, prog, hcur, nb, ch, cw, f"down_blocks.{i}.downsamplers.0.conv", cout,
                                   stride2=True, res2=add, stats=True)
                ai += 1 if with_adds else 0
                ch, cw = (ch + 1) // 2, (cw + 1) // 2
                skips.append((hcur, ch, cw))
                states_down.append(hcur)
        if with_cn:
            # ControlNet: skip_i += residual_i after the whole down path (:1263-1272); h itself is unchanged
            new_skips = []
            for (sk, sh, sw), r in zip(skips, cn_down):
                o = self._buf(plan, *sk.shape)
                prog.add_add(sk, r, o, sk.numel())
                new_skips.append((o, sh, sw))
                if sk is not hcur and self.kind == "unet":
                    self._free(plan, sk)  # the un-summed state has no further reader
            skips = new_skips

        # ---------------- mid (UNetMidBlock2DCrossAttn)
        cm = boc[-1]
        m0 = self._resnet(plan, prog, "mid_block.resnets.0", hcur, None, nb, ch, cw, cm, tproj,
                          out_scale=cfg.mid_block_scale_factor)
        if with_cn:
            self._free(plan, hcur)  # its skip copy lives on in `new_skips`
        m1 = self._transformer(plan, ctxprog, prog, "mid_block.attentions.0", m0, nb, ch, cw, heads, ctx)
        self._free(plan, m0)
        mid_add = cn_mid if with_cn else (add_mid if with_adds else None)
        hcur = self._resnet(plan, prog, "mid_block.resnets.1", m1, None, nb, ch, cw, cm, tproj,
                            out_scale=cfg.mid_block_scale_factor,
                            add=mid_add if self.kind == "unet" else None)
        self._free(plan, m1)
        if with_cn and with_adds:
            hs = self._buf(plan, *hcur.shape)
            prog.add_add(hcur, add_mid, hs, hcur.numel())
            self._free(plan, hcur)
            hcur = hs
        state_mid = hcur

        if self.kind == "controlnet":
            sdev, sstep, sstride = shared.get("scale_dev") or (plan.scale_dev, None, 0)
            if sdev is None:
                sdev = plan.scale_dev = torch.ones(1, dtype=torch.float32, device=self.device)
            # zero-conv outputs: the caller's buffers (`cn_out`), else persistent ones; `cn_res2` (another ControlNet's
            # residuals) is added after the scale, so chained nets leave the running sum in the last net's outputs;
            # `cn_alpha`: constant per-residual factors (guess mode) next to the device scale
            t_down, t_mid = shared.get("cn_out") or ([None] * len(states_down), None)
            r_down, r_mid = shared.get("cn_res2") or ([None] * len(states_down), None)
            a_down, a_mid = shared.get("cn_alpha") or ([1.0] * len(states_down), 1.0)
            outs_down = []
            for k, st in enumerate(states_down):
                c = st.shape[-1]
                o = t_down[k] if t_down[k] is not None else persistent(st.numel() // c, c)
                outs_down.append(self._linear(plan, prog, st, st.numel() // c, f"controlnet_down_blocks.{k}", c,
                                              bias=self.vec(f"controlnet_down_blocks.{k}.bias"), out=o, res2=r_down[k],
                                              alpha=a_down[k], alpha_dev=sdev, alpha_step=sstep, alpha_stride=sstride))
            o = t_mid if t_mid is not None else persistent(state_mid.numel() // cm, cm)
            out_mid = self._linear(plan, prog, state_mid, state_mid.numel() // cm, "controlnet_mid_block",
                                   cm, bias=self.vec("controlnet_mid_block.bias"), out=o, res2=r_mid, alpha=a_mid,
                                   alpha_dev=sdev, alpha_step=sstep, alpha_stride=sstride)
            plan.outputs["down"], plan.outputs["mid"] = outs_down, out_mid
            for st in states_down + [state_mid]:
                self._free(plan, st)
            return plan

        # ---------------- up
        states_up = []
        ui = 0
        capture = self.kind == "brushnet"  # BrushNet's zero-convs read every up state later
        for i, btype in enumerate(cfg.up_block_types):
            cout = list(reversed(boc))[i]
            has_attn = btype == "CrossAttnUpBlock2D"
            for j in range(cfg.layers_per_block + 1):
                skip, sh, sw = skips.pop()
                assert (sh, sw) == (ch, cw), ((sh, sw), (ch, cw))
                rn = f"up_blocks.{i}.resnets.{j}"
                add = next_add(adds_up, ui) if with_adds else None
                prev = hcur
                hcur = self._resnet(plan, prog, rn, hcur, skip.view(nb, ch * cw, skip.shape[-1]), nb, ch, cw, cout,
                                    tproj, add=None if has_attn else add)
                if not capture:
                    self._free(plan, skip)
                    if prev is not state_mid or self.kind == "unet":
                        self._free(plan, prev)
                if has_attn:
                    r_out = hcur
                    hcur = self._transformer(plan, ctxprog, prog, f"up_blocks.{i}.attentions.{j}", hcur, nb, ch, cw,
                                             heads, ctx, add=add)
                    self._free(plan, r_out)
                ui += 1 if with_adds else 0
                # BrushNet captures the state BEFORE the add; BrushNet itself has no adds, so for
                # kind == "brushnet" hcur is exactly the captured tensor
                states_up.append(hcur)
            if i != len(boc) - 1:
                # Upsample2D: nearest to 2x, or to the size of the next skip when the latent is not a multiple
                # of 2^(levels-1) (`upsample_size`, unet_2d_condition.py:1120-1126,1311-1312)
                _, th, tw = skips[-1]
                up = self._buf(plan, nb, th * tw, cout)
                prog.add_upsample_nearest(hcur, up, nb, ch, cw, cout, th, tw)
                if not capture:
                    self._free(plan, hcur)
                ch, cw = th, tw
                add = next_add(adds_up, ui) if with_adds else None
                hcur = self._conv3(plan, prog, up, nb, ch, cw, f"up_blocks.{i}.upsamplers.0.conv", cout, res2=add,
                                   stats=True)
                self._free(plan, up)
                ui += 1 if with_adds else 0
                states_up.append(hcur)

        if self.kind == "brushnet":
            plan.outputs["states"] = (states_down, state_mid, states_up)
            return plan  # zero-convs are appended by `append_brushnet_outputs` (they need the scale)

        # ---------------- out
        gno = self._gn(plan, prog, hcur, None, nb, h * w, "conv_norm_out", cfg.norm_eps, True)
        self._free(plan, hcur)
        eps = persistent(nb, h * w, cfg.out_channels, dtype=torch.float32)
        self._conv3(plan, prog, gno, nb, h, w, "conv_out", cfg.out_channels, out_fp32=True, out=eps)
        self._free(plan, gno)
        plan.outputs["eps"] = eps  # fp32 NHWC [nb, h*w, out_channels]
        return plan

    # ------------------------------------------------------------------ BrushNet zero-convs
    def append_brushnet_outputs(self, plan: Plan, conditioning_scale: float = 1.0, targets=None, scale_dev=None):
        """1x1 zero-convs x conditioning_scale on the 12 + 1 + 15 captured states
        (BrushNet_CA.py:843-845, :861, :900-902, :930-934). `targets` = (down, mid, up) buffer
        lists of a UNet plan (`with_brushnet_adds=True`) to write straight into. `scale_dev` =
        (tensor, step_idx, stride): the scale is multiplied by tensor[*step_idx * stride] on the device, so one
        recorded program serves every `brushnet_conditioning_scale` and the per-step `brushnet_keep` flags
        (pipeline_PowerPaint_Brushnet_CA.py:1369-1376,1403-1409)."""
        states_down, state_mid, states_up = plan.outputs["states"]
        prog = plan.program
        sdev, sstep, sstride = scale_dev or (None, None, 0)

        def zc(st, wname, out):
            c = st.shape[-1]
            M = st.numel() // c
            if out is None:  # read by the caller / by another net's ops: never recycled
                out = torch.empty(M, c, dtype=BF16, device=self.device)
                plan.bytes += out.numel() * 2
            return self._linear(plan, prog, st, M, wname, c, bias=self.vec(wname + ".bias"), alpha=conditioning_scale,
                                out=out, alpha_dev=sdev, alpha_step=sstep, alpha_stride=sstride)
        t_down, t_mid, t_up = targets if targets is not None else (None, None, None)
        outs_down = [zc(st, f"brushnet_down_blocks.{k}", t_down[k] if t_down else None) for k, st in enumerate(states_down)]
        out_mid = zc(state_mid, "brushnet_mid_block", t_mid)
        outs_up = [zc(st, f"brushnet_up_blocks.{k}", t_up[k] if t_up else None) for k, st in enumerate(states_up)]
        plan.outputs["down"], plan.outputs["mid"], plan.outputs["up"] = outs_down, out_mid, outs_up
        plan.outputs["conditioning_scale"] = conditioning_scale
        for st in states_down + [state_mid] + states_up:  # every reader of the captured states is recorded
            self._free(plan, st)

    # ------------------------------------------------------------------ ControlNet cond embedding
    def _build_cond_embedding(self, plan, cond_in, cond_emb, nb, H, W):
        """controlnet_cond_embedding: conv3x3(3->16)+SiLU, [conv+SiLU, conv s2+SiLU] x3, zero conv
        (SURVEY.md App. A.9); independent of t, so it runs once per call, not per step."""
        prog = ops.Program()
        ce = self.cfg.conditioning_embedding_out_channels
        pre = "controlnet_cond_embedding"
        cpad = cond_in.shape[-1]

        def conv(x, name, cout, hh, ww, stride2=False, act=True, out=None, pad_in=None):
            cin = x.shape[-1]
            ho, wo = ((hh + 1) // 2, (ww + 1) // 2) if stride2 else (hh, ww)
            cout_pad = _ceil(cout, 8)
            if out is None:  # own storage: this program runs outside the step program, no recycling across them
                o = torch.zeros(nb, ho * wo, cout_pad, dtype=BF16, device=self.device)
                plan.bytes += o.numel() * 2
            else:
                o = out
            prog.add(ops.gemm_desc(a0=x, w=self.w_conv3(name, pad_in=pad_in or cin), out=o, N_=cout,
                                   a_mode=N.PP_A_CONV3X3_S2 if stride2 else N.PP_A_CONV3X3, c0=cin, nb=nb, h=hh, w_=ww,
                                   bias=self.vec(name + ".bias"), act=N.PP_ACT_SILU if act else N.PP_ACT_NONE,
                                   ldc=cout_pad))
            return o
        x = conv(cond_in, pre + ".conv_in", ce[0], H, W, pad_in=cpad)
        hh, ww = H, W
        for i in range(len(ce) - 1):
            x = conv(x, f"{pre}.blocks.{2 * i}", ce[i], hh, ww)
            x = conv(x, f"{pre}.blocks.{2 * i + 1}", ce[i + 1], hh, ww, stride2=True)
            hh, ww = (hh + 1) // 2, (ww + 1) // 2
        conv(x, pre + ".conv_out", self.cfg.block_out_channels[0], hh, ww, act=False, out=cond_emb)
        return prog
