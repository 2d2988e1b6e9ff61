"""SSIM / MS-SSIM on the fused sm_100a kernel (medical_image_generation_b200.metrics) against the dense algorithm
monai-generative runs (five depthwise cuDNN conv{2,3}d per scale with the full window, fp32), on three workloads:

  a  SSIM, kernel_size 11: 8 reconstruction pairs of 1 x 160 x 160 x 128 (config-5 patch), fp32
  b  all-pairs MS-SSIM (sample diversity), kernel_size 4, 5 scales: 64 volumes of 1 x 128 x 128 x 64 (config 4), bf16,
     2016 pairs (the dense leg computes in fp32 on the same values, 64 pairs per batch)
  c  2-D SSIM, kernel_size 11: 64 pairs of 1 x 256 x 256, fp32

    python tools/ssim_bench.py [--repeats 5] [--json OUT]

Per workload, as one JSON object:
  fused_s / dense_s -- the whole public call ending in a device synchronise (host clock), warmed up, median and best of
                       --repeats; the two legs alternate within each repeat; speedup = dense median / fused median
  kernel_ms         -- CUDA-event time of the SSIM kernel launches alone (inputs already channels-last, the MS-SSIM
                       pyramid already built), averaged over --repeats
  fma / fma_rate    -- multiply-adds of the separable algorithm, from shapes: per scale, pairs x C x valid output voxels
                       x 5 moments x (kd + kh + kw) taps; over kernel_ms. Compared with the FP32 FMA ceiling DERIVED from
                       this run's max SM clock: 148 SMs x 128 lanes x clock (an FMA per lane per cycle), not a data-sheet
                       figure. The per-voxel SSIM arithmetic and the halo rows of the tile are not counted.
  bytes / gbs       -- algorithmic bytes: each operand read once per scale (for b: each of the 64 volumes once per
                       scale, plus writing and reading the pooled pyramid); over kernel_ms, compared with the
                       device-to-device copy bandwidth measured in this run
  bound             -- whichever of the two gives the longer least time; frac_of_bound = that least time / kernel_ms
  gpu               -- name, power limit and max SM clock, read in the same run
There is no CPU path: without a CUDA device the script fails."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from medical_image_generation_b200 import metrics, ops  # noqa: E402

SMS, LANES = 148, 128


def gpu_info(dev) -> dict:
    idx = torch.cuda.current_device() if dev.index is None else dev.index
    q = subprocess.run(["nvidia-smi", f"--id={idx}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().split(",")] + ["?", "?", "?"])[:3]
    return {"name": name if q.returncode == 0 else torch.cuda.get_device_name(dev), "power_limit": power,
            "max_sm_clock": clock}


def copy_gbs(dev) -> float:
    src, dst = torch.empty(1 << 28, device=dev), torch.empty(1 << 28, device=dev)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    return 2 * src.numel() * 4 * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9


# ---- the dense algorithm as monai-generative computes it (fp32, cuDNN depthwise convolutions) ----------------------
def dense_ssim_cs(x, y, win, c1, c2):
    conv = F.conv3d if x.ndim == 5 else F.conv2d
    w = win.expand(x.shape[1], 1, *win.shape).contiguous()
    f = lambda t: conv(t, w, groups=x.shape[1])  # noqa: E731
    mu_x, mu_y, mu_xx, mu_yy, mu_xy = f(x), f(y), f(x * x), f(y * y), f(x * y)
    sx, sy, sxy = mu_xx - mu_x * mu_x, mu_yy - mu_y * mu_y, mu_xy - mu_x * mu_y
    cs = (2 * sxy + c2) / (sx + sy + c2)
    ssim = ((2 * mu_x * mu_y + c1) / (mu_x ** 2 + mu_y ** 2 + c1)) * cs
    return ssim.flatten(1).mean(1), cs.flatten(1).mean(1)


def dense_ms_ssim(x, y, win, weights, c1, c2):
    pool = F.avg_pool3d if x.ndim == 5 else F.avg_pool2d
    vals = []
    for s in range(len(weights)):
        ssim, cs = dense_ssim_cs(x, y, win, c1, c2)
        vals.append(torch.relu(cs))
        x, y = pool(x, kernel_size=2), pool(y, kernel_size=2)
    vals[-1] = torch.relu(ssim)
    w = torch.tensor(weights, device=x.device).view(-1, 1)
    return torch.prod(torch.stack(vals) ** w, dim=0)


def dense_window(taps):
    out = taps[0].double()
    for t in taps[1:]:
        out = out[..., None] * t.double()
    return out.float()


# ---- counts from shapes ---------------------------------------------------------------------------------------------
def fma_per_pair(spatial, C, ks) -> int:
    """Separable algorithm: valid output voxels x C x 5 moments x (sum of the 1-D window lengths)."""
    n = 1
    for s, k in zip(spatial, ks):
        n *= s - k + 1
    return n * C * 5 * sum(ks)


def _timed_pair(fused, dense, repeats):
    f_s, d_s = [], []
    fused(), dense()   # warm-up of every shape of the timed window
    torch.cuda.synchronize()
    for _ in range(repeats):
        for fn, acc in ((fused, f_s), (dense, d_s)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            acc.append(time.perf_counter() - t0)
    return ({"median": statistics.median(f_s), "best": min(f_s)}, {"median": statistics.median(d_s), "best": min(d_s)})


def _event_ms(launch, repeats):
    launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(repeats):
        launch()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / repeats


def _rates(res, fma, nbytes, clock_mhz, copy):
    ms = res["kernel_ms"]
    ceiling = SMS * LANES * clock_mhz * 1e6
    res.update(fma=fma, fma_rate=fma / (ms * 1e-3), fp32_fma_ceiling_derived=ceiling,
               frac_of_fma_ceiling=fma / (ms * 1e-3) / ceiling, bytes=nbytes, gbs=nbytes / (ms * 1e-3) / 1e9,
               frac_of_copy_bw=nbytes / (ms * 1e-3) / 1e9 / copy)
    t_compute, t_bytes = fma / ceiling, nbytes / (copy * 1e9)
    res["bound"] = "fp32_fma" if t_compute >= t_bytes else "bandwidth"
    res["frac_of_bound"] = max(t_compute, t_bytes) / (ms * 1e-3)
    res["speedup"] = res["dense_s"]["median"] / res["fused_s"]["median"]
    return res


def _smooth(shape, g, dev):
    x = torch.rand(shape, generator=g).to(dev)
    k = torch.ones(1, 1, *([5] * (len(shape) - 2)), device=dev) / 5 ** (len(shape) - 2)
    conv = F.conv3d if len(shape) == 5 else F.conv2d
    x = conv(x.flatten(0, 1).unsqueeze(1), k, padding=2).view(shape)
    return (x - x.min()) / (x.max() - x.min())


def workload_ssim(name, shape, ks, dev, repeats, clock, copy):
    g = torch.Generator().manual_seed(0)
    sd = len(shape) - 2
    x = _smooth(shape, g, dev)
    y = (0.8 * x + 0.1 + 0.03 * torch.randn(shape, generator=g).to(dev)).float()
    m = metrics.SSIMMetric(sd, kernel_size=ks)
    win = dense_window(m.taps).to(dev)
    fused = lambda: m(x, y)  # noqa: E731
    dense = lambda: dense_ssim_cs(x, y, win, m.c1, m.c2)  # noqa: E731
    v_f, v_d = fused().view(-1).double(), dense()[0].double()
    f, d = _timed_pair(fused, dense, repeats)
    m.reset()
    pairs = metrics._diagonal_pairs(shape[0], dev)
    ms = _event_ms(lambda: metrics._pair_stats(x, y, pairs, m.taps, m.c1, m.c2), repeats)
    res = {"workload": name, "shape": list(shape), "kernel_size": ks, "dtype": "fp32", "pairs": shape[0],
           "fused_s": f, "dense_s": d, "kernel_ms": ms, "max_abs_diff_vs_dense": (v_f - v_d).abs().max().item()}
    fma = shape[0] * fma_per_pair(shape[2:], shape[1], (ks,) * sd)
    return _rates(res, fma, 2 * x.numel() * 4, clock, copy)


def workload_pairwise(dev, repeats, clock, copy, n=64, shape=(128, 128, 64), ks=4, batch=64):
    g = torch.Generator().manual_seed(1)
    base = _smooth((1, 1) + shape, g, dev)
    own = _smooth((n, 1) + shape, g, dev)
    w = torch.linspace(0.1, 0.9, n, device=dev).view(-1, 1, 1, 1, 1)
    x = (w * base + (1 - w) * own).to(torch.bfloat16)
    m = metrics.MultiScaleSSIMMetric(3, kernel_size=ks)
    I, J = (t.to(dev) for t in torch.triu_indices(n, n, 1))
    P = I.numel()
    xf = x.float()
    win = dense_window(m.taps).to(dev)

    def dense():
        return torch.cat([dense_ms_ssim(xf[I[s:s + batch]], xf[J[s:s + batch]], win, m.weights, m.c1, m.c2)
                          for s in range(0, P, batch)])

    fused = lambda: metrics.pairwise_ms_ssim(x, kernel_size=ks)  # noqa: E731
    v_f, v_d = fused().double(), dense().double()
    f, d = _timed_pair(fused, dense, repeats)
    # kernel time: the five scale launches over the whole pair table on a pyramid built beforehand
    table = torch.stack([I, J], 1).to(torch.int32).contiguous()
    pyr, lvl = [x], x
    for _ in range(len(m.weights) - 1):
        lvl = metrics._pool(lvl)
        pyr.append(lvl)

    def kernels():
        for lv in pyr:
            metrics._pair_stats(lv, lv, table, m.taps, m.c1, m.c2)

    ms = _event_ms(kernels, repeats)
    fma, nbytes = 0, 0
    for s, lv in enumerate(pyr):
        fma += P * fma_per_pair(lv.shape[2:], 1, (ks,) * 3)
        nbytes += lv.numel() * lv.element_size()                          # every volume read once at this scale
        if s:
            nbytes += lv.numel() * 4 + pyr[s - 1].numel() * pyr[s - 1].element_size()   # the pool: read + write
    res = {"workload": "b_pairwise_ms_ssim_k4", "shape": [n, 1, *shape], "kernel_size": ks, "dtype": "bf16",
           "pairs": P, "fused_s": f, "dense_s": d, "kernel_ms": ms,
           "max_abs_diff_vs_dense": (v_f - v_d).abs().max().item(),
           "diversity_mean_ms_ssim": v_f.mean().item()}
    return _rates(res, fma, nbytes, clock, copy)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--json", help="also write the result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ssim_bench needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    info = gpu_info(dev)
    clock = float(info["max_sm_clock"].split()[0])
    copy = copy_gbs(dev)
    with torch.no_grad():
        res = {"gpu": info, "copy_d2d_gbs": copy, "workloads": [
            workload_ssim("a_ssim_k11_3d", (8, 1, 160, 160, 128), 11, dev, args.repeats, clock, copy),
            workload_pairwise(dev, args.repeats, clock, copy),
            workload_ssim("c_ssim_k11_2d", (64, 1, 256, 256), 11, dev, args.repeats, clock, copy)]}
    res["gpu_after"] = gpu_info(dev)
    line = json.dumps(res, indent=1)
    print(line)
    if args.json:
        with open(args.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
