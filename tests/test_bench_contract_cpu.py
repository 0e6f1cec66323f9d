"""CPU tests of the bench.py contract the driver relies on: the reference arm prints ONE JSON line with the agreed keys
(here on a 1-step sample), and the product arm refuses to run without a GPU instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True,
                          text=True, timeout=timeout, env=dict(os.environ, **(env or {})))


def test_reference_arm_prints_one_contract_line():
    # a small net on 128x128 pixels instead of the metric's workload: the line's format is what is checked here, and
    # building + running the SD-1.5-size fp32 net costs ~10 minutes on an 8-vCPU host (the sample string of such a line
    # says that it is not the metric's workload)
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", env={"PP_BENCH_CPU_FORMAT_CHECK": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["metric"] == "512x512 50-step inpaint images/sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert "PP_BENCH_CPU_FORMAT_CHECK=1" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # both arms of one (config, N) carry the same `config` object
    sys.path.insert(0, ROOT)
    import bench

    assert d["config"] == bench.line_config("C2", bench.CONFIGS["C2"], 1)


def test_reference_arm_times_the_loop_of_the_named_config():
    """--config C3 / C5: the CPU arm runs the BrushNet / ControlNet oracle loop, and says so"""
    for name, word in (("C3", "BrushNet"), ("C5", "ControlNet")):
        r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--config", name,
                 env={"PP_BENCH_CPU_FORMAT_CHECK": "1"})
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
        assert d["config"]["name"] == name and word in d["config"]["workload"] and d["value"] > 0
    sys.path.insert(0, ROOT)
    import bench

    assert "BrushNet + UNet" in bench.cpu_sample_text(bench.CONFIGS["C3"])
    assert "1024x1024" in bench.cpu_sample_text(bench.CONFIGS["C4"])


def test_steps_below_one_are_refused():
    """--steps is the number of timed steps of every timed region, so zero timed steps is an error, not a line"""
    r = _run("--steps", "0", timeout=120)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_product_arm_refuses_to_run_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        return  # (on a GPU box the product arm is what `bench.py` itself exercises)
    r = _run("--steps", "1", "--warmup", "0", timeout=120)
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")], "no bench line may come from a CPU run"
    assert "no CPU fallback" in (r.stdout + r.stderr)
