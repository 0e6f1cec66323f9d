#!/usr/bin/env python
"""bench.py — 50-step inpainting throughput of the PowerPaint denoising hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--config C2|C3|C4|C5] [--dump-outputs DIR]   (N > 1: under torchrun)
    python bench.py --impl reference [--gpus N ...]                          CPU arm: the oracle port of the reference

Workloads (BASELINE.json `configs`; every rank runs the per-GPU share, weak scaling):
  C2  PowerPaint-v1 text-guided inpaint, 8 x 512x512 per GPU, UNet batch 16             (default; the metric's config)
  C3  PowerPaint-v2-1 BrushNet object removal, 32 x 512x512 on 8 GPUs = 4 per GPU, BrushNet 8 + UNet 8 per step
  C4  PowerPaint-v1 outpainting, 8 x 1024x1024 on 4 GPUs = 2 per GPU, UNet batch 4, 128x128 latents
  C5  PowerPaint-v1 + ControlNet, 16 x 512x512 on 8 GPUs = 2 per GPU, ControlNet 4 + UNet 4 per step
all 50 DDIM steps, CFG 7.5, bf16 storage / fp32 accumulate, synthetic seeded weights (no checkpoint is reachable
offline) and synthetic image + mask + prompt-embedding batches. One bench "step" = one full 50-step denoise of the
per-GPU batch.

  value  images/s, whole job (sum over GPUs): the denoising loop with inputs already resident in HBM — CUDA-event
         timed, max over ranks.
  e2e    the same metric through the reference-facing pipeline `__call__` with pinned HOST buffers: uint8 images
         and masks + prompt embeddings uploaded by each rank for its own shard, normalised on the device, VAE
         encode, 50 fused steps, VAE decode (all on the repo's kernels), uint8 images gathered to rank 0 (NCCL) and
         read back to the host (output_type="uint8": the device-side form of the uint8 arrays "pil" is built from).
  roofline  tensor-bound: algorithmic FLOPs of one denoising step / mean device time of one recorded step program
         (one CUDA-graph replay), against the measured sustained bf16 peak of MEASURED_PEAKS.json.
  cpu_baseline  the fp32 oracle port of the config's loop on the host cores (bounded sample, fixed thread count);
         `--impl reference` prints the same measurement as its own line, with the same `config` object.
  gpu_library_baseline  the oracle modules in torch bf16 eager (cuDNN / cuBLAS / SDPA: the library path the
         reference reaches through diffusers) on the same GPU, same UNet batch — the practical "reference-GPU" bar.
  parity_spot_check  2 steps of the bench shape against the fp32 oracle (GPU), rel-L2 / cosine; all outputs finite.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "512x512 50-step inpaint images/sec"
UNIT = "images/s"
DDIM_STEPS = 50
GUIDANCE = 7.5
# algorithmic FLOPs of one forward per sample (BASELINE.md section 2)
FLOP_UNET = {64: 0.8034e12, 128: 4.674e12}
FLOP_BRUSHNET = 0.8262e12
FLOP_CONTROLNET = 0.2686e12

CONFIGS = {
    "C2": dict(mode="v1", batch=8, latent=64, flops_per_image_step=2 * FLOP_UNET[64],
               workload="PowerPaint-v1 text-guided inpaint, batch 8 x 512x512 per GPU, 50 DDIM steps, CFG 7.5 "
                        "(UNet batch 16), bf16, synthetic seeded weights (BASELINE.json configs[1])"),
    "C3": dict(mode="brushnet", batch=4, latent=64, flops_per_image_step=2 * (FLOP_UNET[64] + FLOP_BRUSHNET),
               workload="PowerPaint-v2-1 BrushNet object-removal, 32 x 512x512 on 8 GPUs = 4 per GPU (BrushNet batch 8 "
                        "+ UNet batch 8 per step), 50 steps, bf16 (BASELINE.json configs[2])"),
    "C4": dict(mode="v1", batch=2, latent=128, flops_per_image_step=2 * FLOP_UNET[128],
               workload="PowerPaint-v1 outpainting, 8 x 1024x1024 on 4 GPUs = 2 per GPU (UNet batch 4, 128x128 latents), "
                        "50 steps, bf16 (BASELINE.json configs[3])"),
    "C5": dict(mode="controlnet", batch=2, latent=64, flops_per_image_step=2 * (FLOP_UNET[64] + FLOP_CONTROLNET),
               workload="PowerPaint-v1 + ControlNet (canny) inpaint, 16 x 512x512 on 8 GPUs = 2 per GPU (ControlNet batch 4 "
                        "+ UNet batch 4 per step), 50 steps, bf16 (BASELINE.json configs[4])"),
}


def _dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(tflops=float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1467.7))),
                    hbm=float(p.get("hbm_gbs", 6570.6)), src="MEASURED_PEAKS.json (bf16_tflops_sustained)")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback of B200_PROFILING.md (sustained)")


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region"""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append((float(parts[0]), float(parts[1])))
                    for n, v in zip(names, parts[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": sorted(self.reasons)}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": sorted(self.reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------- CPU arm (oracle port)
_CPU_NETS = {}


def cpu_threads() -> int:
    """A FIXED thread count so that every leg of every run reports the same baseline: the physical cores of one
    NUMA node of the host (lscpu), capped at 32 — torch's fp32 conv/GEMM throughput stops scaling (and gets
    noisy) beyond one node. Falls back to half the logical CPUs."""
    try:
        out = subprocess.run(["lscpu"], capture_output=True, text=True, timeout=5).stdout
        kv = {m.group(1).strip(): m.group(2).strip() for m in re.finditer(r"^([^:\n]+):\s*(.+)$", out, re.M)}
        cores = int(kv["Core(s) per socket"]) * int(kv["Socket(s)"])
        nodes = max(1, int(kv.get("NUMA node(s)", "1")))
        n = max(1, cores // nodes)
    except Exception:
        n = max(1, (os.cpu_count() or 2) // 2)
    return max(1, min(n, 32, os.cpu_count() or n))


def _cpu_format_check_only() -> bool:
    """tests/test_bench_contract_cpu.py sets PP_BENCH_CPU_FORMAT_CHECK=1 to check the reference arm's line format in
    seconds: the sample then runs a small net on 128x128 pixels, and the line says so in `sample` (building and
    running the SD-1.5-size fp32 net costs minutes on an 8-vCPU host)."""
    return os.environ.get("PP_BENCH_CPU_FORMAT_CHECK", "0") == "1"


def cpu_sample_text(cfg) -> str:
    if _cpu_format_check_only():
        return ("NOT THE METRIC'S WORKLOAD (PP_BENCH_CPU_FORMAT_CHECK=1: small nets, 1 image at a quarter of the side, "
                "1 of 50 DDIM steps, extrapolated x50)")
    side = 8 * cfg["latent"]
    nets = {"v1": "UNet", "brushnet": "BrushNet + UNet", "controlnet": "ControlNet + UNet"}[cfg["mode"]]
    return (f"fp32 oracle port of the {cfg['mode']} loop ({nets}), 1 image x {side}x{side} (net batch 2, CFG), 1 of 50 DDIM "
            "steps, warm-up pass + best of 2, extrapolated x50")


def cpu_oracle_rate(threads: int, cfg, ddim_steps_sample: int = 1, repeats: int = 2):
    """images/s of the fp32 oracle port of the config's loop (oracle/pipelines.py: v1 / BrushNet / ControlNet) on the host
    cores, extrapolated from a bounded sample: 1 image at the config's resolution (net batch 2 with CFG),
    `ddim_steps_sample` of the 50 steps, best of `repeats` after one untimed warm-up pass (first-touch page faults and
    oneDNN primitive creation otherwise dominate)."""
    from oracle.ddim import DDIMOracle
    from oracle.unet import BrushNetOracle, ControlNetOracle, UNet2DConditionOracle, UNetConfig, build_synthetic

    torch.set_num_threads(threads)
    torch.manual_seed(0)
    tiny = _cpu_format_check_only()
    mk = UNetConfig.tiny if tiny else UNetConfig.sd15
    key = (cfg["mode"], tiny)
    if key not in _CPU_NETS:
        ou = build_synthetic(UNet2DConditionOracle, mk(4 if cfg["mode"] == "brushnet" else 9))
        side = None
        if cfg["mode"] == "brushnet":
            side = build_synthetic(BrushNetOracle, mk(4), seed=99)
        elif cfg["mode"] == "controlnet":
            side = build_synthetic(ControlNetOracle, mk(4), seed=77)
        _CPU_NETS[key] = (ou, side)
    ou, side = _CPU_NETS[key]
    one = dict(cfg, batch=1, latent=cfg["latent"] // 4 if tiny else cfg["latent"])
    kw = resident_inputs(one, torch.device("cpu"), 0, cross=ou.cfg.cross_attention_dim)
    sched = DDIMOracle()

    def one_pass():
        sched.set_timesteps(DDIM_STEPS)
        sched.timesteps = sched.timesteps[:ddim_steps_sample]
        with torch.no_grad():
            return oracle_loop(cfg, ou, side, sched, kw, torch.float32)

    one_pass()  # warm-up, untimed
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        one_pass()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    per_ddim_step = best / ddim_steps_sample
    return 1.0 / (per_ddim_step * DDIM_STEPS), per_ddim_step


def line_config(name: str, cfg, world: int) -> dict:
    """the `config` object of the JSON line: the same for both arms of one (config, N)"""
    B = cfg["batch"]
    return {"workload": cfg["workload"], "name": name, "per_gpu_batch": B, "global_batch": B * world,
            "ddim_steps": DDIM_STEPS, "parallelism": f"batch-sharded x{world}, no collective inside the loop",
            "l2": "working set per step (1.7+ GB weights + activations) exceeds the 126 MB L2"}


def run_reference_arm(args):
    rank, world, _ = _dist_env()
    if rank != 0:
        return 0
    threads = cpu_threads()
    cfg = CONFIGS[args.config]
    vals = []
    for i in range(args.warmup + args.steps):
        v, per = cpu_oracle_rate(threads, cfg, ddim_steps_sample=1, repeats=2 if i >= args.warmup else 1)
        if i >= args.warmup:
            vals.append((v, per))
    v = max(x[0] for x in vals)
    per = min(x[1] for x in vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per * DDIM_STEPS * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": line_config(args.config, cfg, world),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "host_cpus": os.cpu_count(),
                         "sample": cpu_sample_text(cfg)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference's own diffusers pipeline cannot run here (diffusers==0.27.0 absent, no network); "
                "this times the fp32 oracle port of its loop (oracle/) on the host cores of rank 0's box, one bounded "
                "sample per bench step (`cpu_baseline.sample`), `value` and `ms_per_step` extrapolated to 50 DDIM steps",
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------- GPU arm
def build_pipeline(cfg, dev):
    from powerpaint_b200.engine import NetConfig
    from powerpaint_b200.models import BrushNetModel, ControlNetModel, UNet2DConditionModel
    from powerpaint_b200.models.autoencoder_kl import AutoencoderKL
    from powerpaint_b200.pipelines import (StableDiffusionControlNetInpaintPipeline, StableDiffusionInpaintPipeline,
                                           StableDiffusionPowerPaintBrushNetPipeline)
    from powerpaint_b200.schedulers import DDIMScheduler

    vae = AutoencoderKL.synthetic(seed=4321).to(dev)
    mode = cfg["mode"]
    if mode == "brushnet":
        unet = UNet2DConditionModel.synthetic(NetConfig(in_channels=4), seed=1234).to(dev)
        side = BrushNetModel.synthetic(NetConfig(in_channels=4), seed=99).to(dev)
        return StableDiffusionPowerPaintBrushNetPipeline(vae=vae, text_encoder=None, text_encoder_brushnet=None,
                                                         tokenizer=None, unet=unet, brushnet=side,
                                                         scheduler=DDIMScheduler(), safety_checker=None)
    unet = UNet2DConditionModel.synthetic(NetConfig(in_channels=9), seed=1234).to(dev)
    if mode == "controlnet":
        side = ControlNetModel.synthetic(NetConfig(in_channels=4), seed=77).to(dev)
        return StableDiffusionControlNetInpaintPipeline(vae=vae, text_encoder=None, tokenizer=None, unet=unet,
                                                        controlnet=side, scheduler=DDIMScheduler(),
                                                        safety_checker=None)
    return StableDiffusionInpaintPipeline(vae=vae, text_encoder=None, tokenizer=None, unet=unet,
                                          scheduler=DDIMScheduler(), safety_checker=None)


def synth_requests(cfg, seed):
    """host-side synthetic request batch of one rank (SURVEY.md §8d): uint8 RGB images, uint8 masks (centred 25 %
    rectangle; C4: outpainting border = everything outside the centre), prompt embeddings ~ 0.5 N(0,1), and for C5 a
    uint8 edge-like control image."""
    B, L = cfg["batch"], cfg["latent"]
    H = 8 * L
    g = torch.Generator().manual_seed(seed)
    img = torch.randint(0, 256, (B, 3, H, H), generator=g, dtype=torch.uint8)
    mask = torch.zeros(B, 1, H, H, dtype=torch.uint8)
    q = H // 4
    if cfg is CONFIGS["C4"]:
        mask[:] = 255
        mask[:, :, q:3 * q, q:3 * q] = 0
    else:
        mask[:, :, q:3 * q, q:3 * q] = 255
    out = dict(image=img, mask=mask, pe=torch.randn(B, 77, 768, generator=g) * 0.5,
               ne=torch.randn(B, 77, 768, generator=g) * 0.5)
    if cfg["mode"] == "brushnet":
        out["peU"] = torch.randn(2 * B, 77, 768, generator=g) * 0.5
    if cfg["mode"] == "controlnet":
        out["control"] = (torch.rand(B, 3, H, H, generator=g) > 0.9).to(torch.uint8) * 255
    return out


def resident_inputs(cfg, dev, rank, cross: int = 768):
    """device-resident loop inputs for `value` (what the pipeline's preparation would hand to the loop)"""
    B, L = cfg["batch"], cfg["latent"]
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    kw = dict(latents=torch.randn(B, 4, L, L, device=dev, generator=g),
              prompt_embeds=torch.randn(2 * B, 77, cross, device=dev, generator=g) * 0.5)
    mask = torch.zeros(B, 1, L, L, device=dev)
    mask[:, :, L // 4:3 * L // 4, L // 4:3 * L // 4] = 1.0
    ml = torch.randn(B, 4, L, L, device=dev, generator=g)
    if cfg["mode"] == "brushnet":
        cond = torch.cat([ml, mask], 1)
        kw.update(extra=torch.cat([cond, cond]), side_scale=1.0,
                  side_prompt_embeds=torch.randn(2 * B, 77, cross, device=dev, generator=g) * 0.5)
    else:
        kw.update(extra=torch.cat([mask, ml], 1))
    if cfg["mode"] == "controlnet":
        kw.update(side_prompt_embeds=kw["prompt_embeds"], side_scale=0.5,
                  control_image=torch.cat([(torch.rand(B, 3, 8 * L, 8 * L, device=dev, generator=g) > 0.9).float()] * 2))
    return kw


def oracle_nets(cfg, pipe, dev, dtype):
    """the oracle restatement of the bench's nets with the SAME synthetic weights (checker / library baseline)"""
    from oracle.unet import BrushNetOracle, ControlNetOracle, UNet2DConditionOracle, UNetConfig

    cin = pipe.unet.config.in_channels
    ou = UNet2DConditionOracle(UNetConfig.sd15(cin))
    ou.load_state_dict(pipe.unet.state_dict())
    ou = ou.to(dev).to(dtype).eval()
    side = None
    if cfg["mode"] == "brushnet":
        side = BrushNetOracle(UNetConfig.sd15(4))
        side.load_state_dict(pipe.brushnet.state_dict())
    elif cfg["mode"] == "controlnet":
        side = ControlNetOracle(UNetConfig.sd15(4))
        side.load_state_dict(pipe.controlnet.state_dict())
    if side is not None:
        side = side.to(dev).to(dtype).eval()
    return ou, side


def oracle_loop(cfg, ou, side, sched, kw, dtype):
    from oracle.pipelines import loop_brushnet, loop_controlnet, loop_v1

    c = lambda t: t.to(dtype)  # noqa: E731
    if cfg["mode"] == "brushnet":
        return loop_brushnet(ou, side, sched, c(kw["latents"]), c(kw["side_prompt_embeds"]), c(kw["prompt_embeds"]),
                             c(kw["extra"]), GUIDANCE, kw["side_scale"])
    ex = kw["extra"]
    if cfg["mode"] == "controlnet":
        return loop_controlnet(ou, side, sched, c(kw["latents"]), c(kw["prompt_embeds"]), c(ex[:, :1]), c(ex[:, 1:]),
                               c(kw["control_image"]), GUIDANCE, kw["side_scale"])
    return loop_v1(ou, sched, c(kw["latents"]), c(kw["prompt_embeds"]), c(ex[:, :1]), c(ex[:, 1:]), GUIDANCE)


def write_outputs(directory, arrays):
    """`--dump-outputs`: one float32 DIR/<name>.npy per array, so that two builds can be compared output for output"""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.numpy().astype(np.float32))


def run_gpu_arm(args):
    rank, world, local = _dist_env()
    if world != args.gpus and world == 1 and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun with {args.gpus} ranks", file=sys.stderr)
        return 2
    if not torch.cuda.is_available():
        print("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)",
              file=sys.stderr)
        return 2
    cfg = CONFIGS[args.config]
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    from powerpaint_b200 import _native

    assert _native.lib().pp_device_supported() == 1, "bench needs an sm_100 (B200) device"
    pipe = build_pipeline(cfg, dev)
    den = pipe.denoiser()
    sched = pipe.scheduler
    sched.set_timesteps(DDIM_STEPS)
    coef = sched.step_coefficients()
    B, L = cfg["batch"], cfg["latent"]
    H = 8 * L
    kw = resident_inputs(cfg, dev, rank)

    def loop_once(ts=None, cf=None):
        return den.run(timesteps=sched.timesteps if ts is None else ts, coef=coef if cf is None else cf,
                       guidance_scale=GUIDANCE, **kw)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        out = loop_once()
    assert torch.isfinite(out).all(), "non-finite latents after warm-up"
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record()
        for _ in range(args.steps):
            out = loop_once()
        e1.record()
        barrier()
    assert torch.isfinite(out).all(), "non-finite latents in the timed region"
    dump = {"latents": out.float().cpu()} if args.dump_outputs and rank == 0 else None
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = B * world * args.steps / (ms_max / 1e3)
    launches_per_ddim = den.launches_per_step

    # ---- per-step program time for the roofline (events around each graph replay)
    st = next(reversed(den._cache.values()))
    torch.cuda.synchronize()
    with torch.cuda.stream(den._stream):
        st["step_idx"].zero_()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(DDIM_STEPS + 1)]
        evs[0].record()
        for i in range(DDIM_STEPS):
            st["program"].launch()
            evs[i + 1].record()
    torch.cuda.synchronize()
    step_ms = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(5, DDIM_STEPS - 5))
    step_mean = sum(step_ms) / len(step_ms)
    flops_step = cfg["flops_per_image_step"] * B
    pk = _peaks()
    achieved = flops_step / (step_mean / 1e3) / 1e12
    plan_bytes = st["bytes"]

    # ---- e2e through the public pipeline API: pinned host buffers -> ... -> decoded uint8 images on the host
    req = synth_requests(cfg, seed=rank)
    host = {k: v.pin_memory() for k, v in req.items()}
    stage = {k: torch.empty_like(v, device=dev) for k, v in req.items()}
    out_host = torch.empty(B * world, H, H, 3, dtype=torch.uint8).pin_memory() if rank == 0 else None

    def e2e_once():
        for k in host:  # every rank uploads its own shard (no funnel through rank 0)
            stage[k].copy_(host[k], non_blocking=True)
        common = dict(image=stage["image"], mask=stage["mask"], prompt_embeds=stage["pe"],
                      negative_prompt_embeds=stage["ne"], height=H, width=H, num_inference_steps=DDIM_STEPS,
                      guidance_scale=GUIDANCE, generator=torch.Generator().manual_seed(rank), output_type="uint8")
        if cfg["mode"] == "brushnet":
            res = pipe(prompt_embedsU=stage["peU"], brushnet_conditioning_scale=1.0, **common).images
        elif cfg["mode"] == "controlnet":
            res = pipe(control_image=stage["control"], controlnet_conditioning_scale=0.5, **common).images
        else:
            res = pipe(**common).images
        if dist is not None:
            from powerpaint_b200.parallel import gather_images

            res = gather_images(res)
        if rank == 0:
            out_host.copy_(res, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return out_host

    e2e_once()
    e2e_once()
    barrier()
    k_e2e = args.steps
    t0 = time.perf_counter()
    for _ in range(k_e2e):
        e2e_once()
    barrier()
    dt = time.perf_counter() - t0
    if dump is not None:  # rank 0's own shard: the first B of the gathered images
        dump["images"] = out_host[:B].float()
        write_outputs(args.dump_outputs, dump)
    tt = torch.tensor([dt], device=dev)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_value = B * world * k_e2e / float(tt.item())
    h2d = sum(v.numel() * v.element_size() for v in req.values()) * world
    d2h = B * world * 3 * H * H

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": line_config(args.config, cfg, world),
            "detail": {"ms_per_ddim_step": step_mean, "plan_activation_bytes": int(plan_bytes)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "calls_timed": k_e2e,
                    "includes": "per-rank H2D of uint8 image/mask + prompt embeddings from pinned host memory, "
                                "on-device normalisation, VAE encode, 50 fused steps, VAE decode, uint8 images "
                                + ("gathered to rank 0 over NCCL, " if world > 1 else "") + "D2H into pinned memory"},
            "gpu_launches": int(launches_per_ddim * DDIM_STEPS * args.steps),
            "clocks": clocks.summary(),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s",
                         "frac": achieved / pk["tflops"], "traffic": None, "peak_source": pk["src"] + ", of measured",
                         "kernel": "one denoising-step program (side net + UNet forward + CFG/DDIM), "
                                   f"{launches_per_ddim} launches replayed as one CUDA graph",
                         "flops_per_launch": flops_step, "ms_per_launch": step_mean},
        }
        tr = os.path.join(ROOT, "profiles", "r02_step_traffic.json")
        if os.path.exists(tr):  # dram bytes of one step program from the committed ncu capture of this build
            with open(tr) as f:
                tj = json.load(f)
            if tj.get("config") == args.config:
                line["roofline"]["traffic"] = tj.get("dram_bytes_per_step")
                line["roofline"]["traffic_source"] = tj.get("source")
    # ---- checker and baselines (rank 0, single-GPU runs only: they are not part of the timed regions)
    if rank == 0 and world == 1 and not args.no_baselines:
        from oracle.ddim import DDIMOracle

        ou, oside = oracle_nets(cfg, pipe, dev, torch.float32)
        so = DDIMOracle()
        so.set_timesteps(DDIM_STEPS)
        so.timesteps = so.timesteps[:2]
        ts2 = sched.timesteps[:2]
        ref = oracle_loop(cfg, ou, oside, so, kw, torch.float32)
        got = loop_once(ts2, sched.step_coefficients(ts2))
        rel = ((got - ref).norm() / ref.norm()).item()
        cos = torch.nn.functional.cosine_similarity(got.flatten(), ref.flatten(), dim=0).item()
        line["parity_spot_check"] = {"steps": 2, "rel_l2": rel, "cosine": cos, "finite": bool(torch.isfinite(got).all()),
                                     "against": "fp32 oracle loop on the GPU, bench shape and inputs"}
        assert torch.isfinite(got).all() and rel < 5e-2, f"bench-shape parity spot check failed: rel-L2 {rel}"
        # library baseline: the same oracle modules in bf16 eager, 3 steps timed after 2 warm-up steps
        ou = ou.to(torch.bfloat16)
        oside = oside.to(torch.bfloat16) if oside is not None else None
        so.set_timesteps(DDIM_STEPS)
        so.timesteps = so.timesteps[:2]
        oracle_loop(cfg, ou, oside, so, kw, torch.bfloat16)
        so.set_timesteps(DDIM_STEPS)
        so.timesteps = so.timesteps[:3]
        torch.cuda.synchronize()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        oracle_loop(cfg, ou, oside, so, kw, torch.bfloat16)
        b1.record()
        torch.cuda.synchronize()
        lib_ms = b0.elapsed_time(b1) / 3
        line["gpu_library_baseline"] = {
            "value": B / (lib_ms * DDIM_STEPS / 1e3), "unit": UNIT, "ms_per_ddim_step": lib_ms,
            "kind": "torch_eager_restatement",
            "what": "oracle modules in torch bf16 eager (cuDNN / cuBLAS / SDPA), same nets, UNet batch and inputs, "
                    "3 DDIM steps timed, loop only"}
        del ou, oside
        torch.cuda.empty_cache()
        th = cpu_threads()
        cpu_v, cpu_per = cpu_oracle_rate(th, cfg, ddim_steps_sample=1, repeats=2)
        line["cpu_baseline"] = {"value": cpu_v, "unit": UNIT, "cores": th, "kind": "port", "host_cpus": os.cpu_count(),
                                "sample": cpu_sample_text(cfg) + f" ({cpu_per:.2f} s per DDIM step)"}
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--no-baselines", action="store_true",
                    help="skip the parity spot check and the CPU / library baselines (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32, "
                         "rank 0): latents.npy = the denoising loop's final latents [B,4,h,w], images.npy = the e2e "
                         "pipeline call's uint8 images [B,H,W,3] as float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
