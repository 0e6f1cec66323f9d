"""Per-step device time of the fused ControlNet step with one and two ControlNets, each with and without guess mode, at
the C5 per-GPU shape (2 images at 512x512, DDIM 50 steps, CFG 7.5, synthetic SD-1.5 weights). Developer/profile script,
not the judged bench.

    python profiles/bench_controlnet_multi.py [--steps 50] [--rounds 3] [--out FILE]

Method: one warm-up call per variant (records the plan and captures the graph), then per round and variant one timed
call of `--steps` graph replays between CUDA events; the variants alternate within a round so that drift on a shared
host spreads over all of them. Reported: the median over rounds of ms per step, images/s, launches per step and
achieved TFLOP/s with the algorithmic FLOPs of bench.py (FLOP_UNET / FLOP_CONTROLNET; a guess-mode ControlNet runs at
batch B, the UNet at 2B). The card name and power limit are read in the same run and printed beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import FLOP_CONTROLNET, FLOP_UNET  # noqa: E402
from powerpaint_b200.denoise import FusedDenoiser  # noqa: E402
from powerpaint_b200.engine import NetConfig  # noqa: E402
from powerpaint_b200.models import ControlNetModel, MultiControlNetModel, UNet2DConditionModel  # noqa: E402
from powerpaint_b200.schedulers import DDIMScheduler  # noqa: E402

B, LAT, GUIDANCE = 2, 64, 7.5
VARIANTS = [("one_controlnet", 1, False), ("two_controlnets", 2, False), ("guess_one", 1, True), ("guess_two", 2, True)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def flops_per_step(n_nets, guess):
    """algorithmic FLOPs of one fused step: UNet at 2B, each ControlNet at 2B (B in guess mode)"""
    return 2 * B * FLOP_UNET[LAT] + n_nets * (B if guess else 2 * B) * FLOP_CONTROLNET


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda")
    unet = UNet2DConditionModel.synthetic(NetConfig(in_channels=9), seed=1234).to(dev)
    nets = MultiControlNetModel([ControlNetModel.synthetic(NetConfig(in_channels=4), seed=s).to(dev) for s in (77, 78)])
    sched = DDIMScheduler()
    sched.set_timesteps(args.steps)
    ts = sched.timesteps
    g = torch.Generator(device=dev).manual_seed(0)
    lat = torch.randn(B, 4, LAT, LAT, device=dev, generator=g)
    emb = torch.randn(2 * B, 77, 768, device=dev, generator=g) * 0.5
    extra = torch.randn(B, 5, LAT, LAT, device=dev, generator=g)
    ctrls = [torch.rand(B, 3, 8 * LAT, 8 * LAT, device=dev, generator=g) for _ in range(2)]
    dens = {name: FusedDenoiser(unet, nets, "controlnet") for name, _, _ in VARIANTS}
    single = FusedDenoiser(unet, nets.nets[0], "controlnet")  # the plain single-ControlNet path, as bench.py C5 runs it

    def kw(n, guess):
        imgs = [c if guess else torch.cat([c] * 2) for c in ctrls[:n]]
        return dict(latents=lat, prompt_embeds=emb, side_prompt_embeds=emb, control_image=imgs, timesteps=ts,
                    coef=sched.step_coefficients(ts), guidance_scale=GUIDANCE, extra=extra, side_scale=[0.5] * n,
                    guess_mode=guess)

    runs = {name: (dens[name], kw(n, guess)) for name, n, guess in VARIANTS}
    k1 = kw(1, False)
    runs["single_controlnet_model"] = (single, dict(k1, control_image=k1["control_image"][0], side_scale=0.5,
                                                    guess_mode=False))
    for den, k in runs.values():
        den.run(**k)  # warm-up: plan, graph capture
    torch.cuda.synchronize()
    times = {name: [] for name in runs}
    for _ in range(args.rounds):
        for name, (den, k) in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            den.run(**k)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)
    dev_name = card()
    res = dict(card=dev_name, shape=f"{B} x 512x512, DDIM {args.steps} steps, CFG {GUIDANCE}", rounds=args.rounds,
               variants={})
    spec = {name: (n, guess) for name, n, guess in VARIANTS}
    spec["single_controlnet_model"] = (1, False)
    for name, ms in times.items():
        ms_med = sorted(ms)[len(ms) // 2]
        n, guess = spec[name]
        res["variants"][name] = dict(ms_per_step=round(ms_med, 3), ms_all=[round(v, 3) for v in ms],
                                     images_per_s=round(B / (ms_med * args.steps / 1e3), 3),
                                     launches_per_step=runs[name][0].launches_per_step,
                                     tflops_achieved=round(flops_per_step(n, guess) / (ms_med / 1e3) / 1e12, 1))
        print(f"{name:24s} {ms_med:7.3f} ms/step  {res['variants'][name]['images_per_s']:6.2f} images/s  "
              f"{res['variants'][name]['launches_per_step']:5d} launches/step  "
              f"{res['variants'][name]['tflops_achieved']:6.1f} TFLOP/s", flush=True)
    print("card:", dev_name)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
