"""DDPM likelihood (`DiffusionInferer.get_likelihood`) of BASELINE config-4 volumes (1 x 128 x 128 x 64, the bench.py
sampling model in bf16), against `sample` over the same timesteps, plus the fused bound-term kernel alone.

    python tools/likelihood_bench.py [--steps 50] [--repeats 3] [--json OUT]

Reports, as one JSON object:
  likelihood -- per batch B in (1, 4): the first --steps timesteps of the 1000-step schedule through get_likelihood with
                cuda_graph=True and False, alternating in the same process with `sample` (cuda_graph=True) over the same
                timesteps; ms per timestep (median and best of --repeats) and the volumes per minute a full 1000-step
                bound implies. The difference to `sample` is the per-step cost of the bound against the forward.
  kernel     -- mig_ddpm_vlb_term with and without the map, and upstream's ATen composition of the same term (about 20
                elementwise kernels and a mean), on fp32 and bf16 tensors of >= 64 MB, CUDA-event timed, every launch
                on a different buffer of a pool larger than L2; GB/s from the algorithmic bytes and their fraction of
                the device-to-device copy bandwidth measured in the same run
  gpu        -- name, power limit and max SM clock, read in the same run
There is no CPU fallback: without a CUDA device the script fails."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
import medical_image_generation_b200 as mig  # noqa: E402
from ddim_sample_bench import gpu_info  # noqa: E402
from medical_image_generation_b200 import ops, planner  # noqa: E402


def _timed(fn) -> float:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def _summary(secs, n) -> dict:
    med, best = statistics.median(secs), min(secs)
    return {"ms_per_step": 1e3 * med / n, "ms_per_step_min": 1e3 * best / n,
            "volumes_per_min_1000_steps_per_sample": 60.0 / (med / n * 1000), "sec_all": secs}


def likelihood(dev, n, repeats) -> dict:
    torch.manual_seed(7)
    model = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**bench.SAMPLING_CFG, compute_dtype=torch.bfloat16))
    model = model.to(dev).eval()
    s = mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS)
    s.noise_mode = "device"
    s.timesteps = s.timesteps[:n]
    inf = mig.DiffusionInferer(s)
    out = {"steps_timed": n}
    for B in (1, 4):
        g = torch.Generator().manual_seed(42)
        x0 = (torch.rand((B, *bench.VOLUME), generator=g) * 2 - 1).to(dev)
        noise = torch.randn((B, *bench.VOLUME), generator=g).to(dev)
        runs = {
            "likelihood_graph": lambda: inf.get_likelihood(x0, model, noise=noise, cuda_graph=True),
            "likelihood_eager": lambda: inf.get_likelihood(x0, model, noise=noise, cuda_graph=False),
            "sample_graph": lambda: inf.sample(noise, model, s, verbose=False, cuda_graph=True),
        }
        for fn in runs.values():                                           # warm-up
            fn()
        secs = {k: [] for k in runs}
        for _ in range(repeats):                                           # alternate
            for k, fn in runs.items():
                secs[k].append(_timed(fn))
        res = {k: _summary(v, n) for k, v in secs.items()}
        for k in ("likelihood_graph", "likelihood_eager"):
            res[k]["vs_sample_graph"] = res[k]["ms_per_step"] / res["sample_graph"]["ms_per_step"]
            res[k]["volumes_per_min_1000_steps"] = B * res[k]["volumes_per_min_1000_steps_per_sample"]
        total = inf.get_likelihood(x0, model, noise=noise, cuda_graph=True)
        if not torch.isfinite(total).all():
            raise RuntimeError("the bound is not finite")
        out[f"B{B}"] = res
        del x0, noise
    del model
    torch.cuda.empty_cache()
    return out


def aten_term(s, m, xt, x0, t):
    """Upstream's tensor composition of one t > 0 term and its per-sample mean (fp32 math on the stored tensors)."""
    acp = s.alphas_cumprod
    a, ap = acp[t], acp[t - 1]
    m, xt, x0 = m.float(), xt.float(), x0.float()
    x0h = ((xt - (1 - a) ** 0.5 * m) / a ** 0.5).clamp(-1, 1)
    c0 = float((ap ** 0.5 * s.betas[t]) / (1 - a))
    ct = float(s.alphas[t] ** 0.5 * (1 - ap) / (1 - a))
    mu_p = c0 * x0h + ct * xt
    mu_q = c0 * x0 + ct * xt
    lv = torch.log(s._get_variance(t))
    kl = 0.5 * (-1.0 + lv - lv + torch.exp(lv - lv) + ((mu_q - mu_p) ** 2) * torch.exp(-lv))
    return kl.view(kl.shape[0], -1).mean(1)


def kernel(dev, reps=6) -> dict:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(launch, nbytes, r=reps):
        launch(0)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(2):
            for i in range(r):
                launch(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / (2 * r)
        return {"avg_launch_ms": ms, "algorithmic_bytes": nbytes, "gbs": nbytes / (ms * 1e-3) / 1e9}

    src = [torch.empty(1 << 28, device=dev) for _ in range(2)]
    dst = [torch.empty(1 << 28, device=dev) for _ in range(2)]
    copy = timed(lambda i: dst[i % 2].copy_(src[i % 2]), 2 * src[0].numel() * 4)
    del src, dst
    out = {"copy_d2d": copy}
    s = mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS)
    B = 4
    for dtype, numel in ((torch.float32, 16 * 128 * 128 * 64), (torch.bfloat16, 32 * 128 * 128 * 64)):
        es = torch.finfo(dtype).bits // 8
        shape = (B, numel // B)
        m, xt, x0 = ([torch.randn(shape, device=dev).to(dtype) for _ in range(reps)] for _ in range(3))
        ts = torch.full((B,), 500, dtype=torch.int64, device=dev)
        total = torch.zeros(B, dtype=torch.float64, device=dev)
        kl = torch.empty(shape, dtype=torch.float32, device=dev)
        ws = s._vlb_workspace(m[0])
        tag = "fp32" if dtype == torch.float32 else "bf16"
        mb = numel * es / 2 ** 20
        for name, kmap in (("no_map", None), ("map", kl)):
            nb = 3 * numel * es + (numel * 4 if kmap is not None else 0)
            r = timed(lambda i: s._vlb_term(m[i], ts, xt[i], x0[i], total, ws, kmap), nb)
            r["tensor_mb"] = mb
            out[f"vlb_term_{tag}_{name}"] = r
        r = timed(lambda i: aten_term(s, m[i], xt[i], x0[i], 500), 3 * numel * es, r=2)
        r["tensor_mb"] = mb
        out[f"aten_term_{tag}"] = r
        del m, xt, x0, kl
        torch.cuda.empty_cache()
    for name, r in out.items():
        if name != "copy_d2d":
            r["frac_of_measured_copy"] = r["gbs"] / copy["gbs"]
    for tag in ("fp32", "bf16"):
        out[f"aten_over_fused_{tag}"] = out[f"aten_term_{tag}"]["avg_launch_ms"] / \
            out[f"vlb_term_{tag}_no_map"]["avg_launch_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--json", help="also write the result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("likelihood_bench needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    res = {"gpu": gpu_info(dev), "kernel": kernel(dev), "likelihood": likelihood(dev, args.steps, args.repeats)}
    res["gpu_after"] = gpu_info(dev)
    line = json.dumps(res)
    print(line)
    if args.json:
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
