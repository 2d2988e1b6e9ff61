"""DDIM few-step sampling of BASELINE config 4 (1 x 128 x 128 x 64 volumes, the bench.py sampling model in bf16) against
1000-step DDPM, through the public path: `DiffusionInferer.sample(..., cuda_graph=True)` with the step noise drawn on
the device. Also times the fused `ddim_step` kernel alone and relates it to the HBM bandwidth measured in the same run.

    python tools/ddim_sample_bench.py [--steps 50,100,250] [--repeats 5] [--json OUT]

Reports, as one JSON object:
  sampling  -- per DDIM step count n: wall time of one whole n-step volume (graph capture included, as a user pays it),
               ms per reverse step and volumes/min (median and best of --repeats); DDPM timed over the first n steps of
               its 1000-step schedule in the same way, alternating with DDIM, giving its ms per step and the 1000-step
               volumes/min it implies
  kernels   -- ddim_step (and ddpm_step for comparison) on fp32 and bf16 tensors of >= 64 MB each, CUDA-event timed,
               every launch on a different buffer of a pool larger than L2; GB/s from the algorithmic bytes, and its
               fraction of the device-to-device copy bandwidth measured here and of the 7.7 TB/s data-sheet figure
  gpu       -- name, power limit and max SM clock, read in the same run
There is no CPU fallback: without a CUDA device the script fails."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import medical_image_generation_b200 as mig  # noqa: E402
from medical_image_generation_b200 import _lib, ops, planner  # noqa: E402

DATASHEET_HBM_GBS = 7700.0   # HGX B200 data sheet, one GPU


def gpu_info(dev) -> dict:
    idx = torch.cuda.current_device() if dev.index is None else dev.index
    q = subprocess.run(["nvidia-smi", f"--id={idx}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().split(",")] + ["?", "?", "?"])[:3]
    return {"name": name if q.returncode == 0 else torch.cuda.get_device_name(dev), "power_limit": power,
            "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(dev)}


def time_sample(inf, model, sched, noise_host, dev) -> float:
    """Seconds for one volume (host clock around work that ends in a device synchronise): H2D of the noise, the
    reverse steps over `sched.timesteps`, D2H of the result."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vol = inf.sample(noise_host.to(dev, non_blocking=True), model, sched, verbose=False, cuda_graph=True).to("cpu")
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    if not torch.isfinite(vol).all():
        raise RuntimeError("sampled volume is not finite")
    return sec


def _summary(secs, n) -> dict:
    med, best = statistics.median(secs), min(secs)
    return {"sec_per_volume": med, "sec_per_volume_min": best, "ms_per_step": 1e3 * med / n,
            "ms_per_step_min": 1e3 * best / n, "sec_all": secs}


def sampling(dev, steps, repeats) -> dict:
    torch.manual_seed(7)
    model = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**bench.SAMPLING_CFG, compute_dtype=torch.bfloat16))
    model = model.to(dev).eval()
    noise_host = torch.randn((1, *bench.VOLUME), generator=torch.Generator().manual_seed(42)).pin_memory()
    ddim = mig.DDIMScheduler(**planner.LDM_SCHEDULER_KWARGS)
    ddpm = mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS)
    for s in (ddim, ddpm):
        s.noise_mode = "device"
    ddpm.set_timesteps(1000)
    full = ddpm.timesteps
    inf = mig.DiffusionInferer(ddim)
    ddim.set_timesteps(10)                                                # warm-up: workspaces, capture path
    time_sample(inf, model, ddim, noise_host, dev)
    ddpm.timesteps = full[:10]
    time_sample(inf, model, ddpm, noise_host, dev)
    out = {}
    for n in steps:
        ddim.set_timesteps(n)
        ddpm.timesteps = full[:n]
        a, b = [], []
        for _ in range(repeats):                                          # alternate the two schedulers
            a.append(time_sample(inf, model, ddim, noise_host, dev))
            b.append(time_sample(inf, model, ddpm, noise_host, dev))
        da, dp = _summary(a, n), _summary(b, n)
        da["volumes_per_min"] = 60.0 / da["sec_per_volume"]
        dp["volumes_per_min_1000_steps"] = 60.0 / (dp["ms_per_step"] * 1000 / 1e3)
        out[f"ddim_{n}"] = {"steps": n, **da, "ddpm_same_window": {"steps_timed": n, **dp}}
    del model
    torch.cuda.empty_cache()
    return out


def kernels(dev, reps=6) -> dict:
    call, ptr = _lib.call, ops._ptr
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(launch, nbytes):
        launch(0)
        torch.cuda.synchronize()
        e0.record()
        for r in range(2):
            for i in range(reps):
                launch(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / (2 * reps)
        return {"avg_launch_ms": ms, "algorithmic_bytes": nbytes, "gbs": nbytes / (ms * 1e-3) / 1e9}

    # device-to-device copy over a 1 GiB pool per direction: the bandwidth this card reaches in this run
    src = [torch.empty(1 << 28, device=dev) for _ in range(2)]
    dst = [torch.empty(1 << 28, device=dev) for _ in range(2)]
    copy = timed(lambda i: dst[i % 2].copy_(src[i % 2]), 2 * src[0].numel() * 4)
    del src, dst
    out = {"copy_d2d": copy}
    ddim = mig.DDIMScheduler(**planner.LDM_SCHEDULER_KWARGS)
    ddim.set_timesteps(50)
    k = ddim.step_coefficients(500, 1.0)
    ddpm = mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS).step_coefficients(500)
    for dtype, numel in ((torch.float32, 16 * 128 * 128 * 64), (torch.bfloat16, 32 * 128 * 128 * 64)):
        es = torch.finfo(dtype).bits // 8
        m, x, z = ([torch.randn(numel, device=dev).to(dtype) for _ in range(reps)] for _ in range(3))
        prev, x0 = torch.empty_like(m[0]), torch.empty_like(m[0])
        dt = ops._dt(m[0])
        tag = "fp32" if dtype == torch.float32 else "bf16"
        mb = numel * es / 2 ** 20
        for eta, sig in (("eta1", k["sigma"]), ("eta0", 0.0)):
            nb = (5 if sig else 4) * numel * es
            r = timed(lambda i: call("mig_ddim_step", dt, ptr(m[i]), ptr(x[i]), ptr(z[i]) if sig else None, ptr(prev),
                                     ptr(x0), numel, k["sqrt_acp"], k["sqrt_one_minus_acp"], k["sqrt_acp_prev"],
                                     k["dir_coef"], sig, 0, 1, ops._stream()), nb)
            r["tensor_mb"] = mb
            out[f"ddim_step_{tag}_{eta}"] = r
        r = timed(lambda i: call("mig_ddpm_step", dt, ptr(m[i]), ptr(x[i]), ptr(z[i]), ptr(prev), ptr(x0), numel,
                                 ddpm["sqrt_acp"], ddpm["sqrt_one_minus_acp"], ddpm["c0"], ddpm["ct"], ddpm["sigma"], 0, 1,
                                 ops._stream()), 5 * numel * es)
        r["tensor_mb"] = mb
        out[f"ddpm_step_{tag}"] = r
        del m, x, z, prev, x0
    for name, r in out.items():
        if name != "copy_d2d":
            r["frac_of_measured_copy"] = r["gbs"] / copy["gbs"]
            r["frac_of_datasheet"] = r["gbs"] / DATASHEET_HBM_GBS
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", default="50,100,250")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--json", help="also write the result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ddim_sample_bench needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    res = {"gpu": gpu_info(dev), "kernels": kernels(dev),
           "sampling": sampling(dev, [int(s) for s in args.steps.split(",")], args.repeats)}
    res["gpu_after"] = gpu_info(dev)
    line = json.dumps(res, indent=1)
    print(line)
    if args.json:
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
