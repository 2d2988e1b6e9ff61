"""Shared helpers for the parity tests (TEST CODE: may import oracle/)."""
import torch

FP32_TOL = 1e-4   # north_star: per-block fp32 outputs within 1e-4 relative error
BF16_TOL = 2e-2   # north_star: bf16 within 2e-2


def rel_err(got, want, floor=1e-30):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).norm() / want.norm().clamp_min(floor))


def bf16_round(t):
    return t.to(torch.bfloat16).to(torch.float32)


def tol_for(dtype):
    return FP32_TOL if dtype == torch.float32 else BF16_TOL


def local_errors(got, want) -> dict:
    """Relative errors of `got` against `want`, both laid out (N, C, *spatial) (a 1-D tensor is one sample of C
    channels), computed in fp64 on `want`'s device:
      glob -- ||got - want|| / ||want|| over the whole tensor (what `rel_err` measures);
      row  -- per voxel: the error norm over the channels of one (n, *spatial) position, divided by the larger of that
              position's norm and the rms of all positions' norms, worst position in `row_at`;
      col  -- per channel: the same over all (n, *spatial) of one channel, worst channel in `col_at`.
    A global ratio averages an error confined to a fraction f of the tensor down by sqrt(f) (one 64-voxel box of an
    8 x 256 x 24^3 activation: f = 5.8e-4); the per-voxel and per-channel ratios do not."""
    w = want.detach().to(torch.float64)
    g = got.detach().to(device=w.device, dtype=torch.float64)
    if tuple(g.shape) != tuple(w.shape):
        raise AssertionError(f"shape {tuple(g.shape)} != reference shape {tuple(w.shape)}")
    if w.ndim == 1:
        g, w = g[None], w[None]
    e = g - w
    glob = float(e.norm() / w.norm().clamp_min(1e-30))
    ev, wv = e.pow(2).sum(1).sqrt(), w.pow(2).sum(1).sqrt()                 # (N, *spatial)
    row = ev / torch.maximum(wv, wv.pow(2).mean().sqrt()).clamp_min(1e-30)
    dims = (0,) + tuple(range(2, w.ndim))
    ec, wc = e.pow(2).sum(dims).sqrt(), w.pow(2).sum(dims).sqrt()           # (C,)
    col = ec / torch.maximum(wc, wc.pow(2).mean().sqrt()).clamp_min(1e-30)
    at = torch.unravel_index(row.argmax(), tuple(row.shape))
    return {"glob": glob, "row": float(row.max()), "row_at": tuple(int(i) for i in at),
            "col": float(col.max()), "col_at": int(col.argmax())}


def local_failure(errs: dict, *, glob, row, col, what) -> "str | None":
    """The failure message for `local_errors` output against the three bars, or None when all three hold."""
    if errs["glob"] <= glob and errs["row"] <= row and errs["col"] <= col:
        return None
    return (f"{what}: global {errs['glob']:.3e} (bar {glob:.1e}), worst voxel (n, *spatial) {errs['row_at']} "
            f"{errs['row']:.3e} (bar {row:.1e}), worst channel {errs['col_at']} {errs['col']:.3e} (bar {col:.1e})")


def assert_close_local(got, want, *, glob, row, col, what) -> dict:
    """Fails when the global, the worst per-voxel or the worst per-channel relative error exceeds its bar; the message
    names the worst voxel as (n, d, h, w) and the worst channel, i.e. the box or tile to look at. Returns the errors."""
    errs = local_errors(got, want)
    msg = local_failure(errs, glob=glob, row=row, col=col, what=what)
    assert msg is None, msg
    return errs


def f32(x: float) -> float:
    """`x` rounded to fp32: the value a hyperparameter has after crossing the C ABI as a float."""
    return float(torch.tensor(x, dtype=torch.float32))


def clip_adamw_reference(params, grads, exp_avgs, exp_avg_sqs, step, *, lr, betas, eps, weight_decay, max_norm):
    """fp64 restatement of torch.nn.utils.clip_grad_norm_(max_norm) followed by ONE torch.optim.AdamW step (decoupled
    weight decay, bias corrections 1 - beta**step). Every tensor is taken to float64; max_norm 0 / None: no clipping.
    Returns (params, exp_avgs, exp_avg_sqs, total_norm, clip_coef) after the step (new float64 tensors). As in torch, the
    clamp of the clip coefficient keeps a NaN: a NaN in any gradient makes every parameter NaN."""
    d = lambda ts: [t.detach().to(torch.float64) for t in ts]  # noqa: E731
    ps, gs, ms, vs = d(params), d(grads), d(exp_avgs), d(exp_avg_sqs)
    total = torch.stack([g.pow(2).sum() for g in gs]).sum().sqrt()
    coef = torch.ones((), dtype=torch.float64)
    if max_norm:
        coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    b1, b2 = betas
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    out_p, out_m, out_v = [], [], []
    for p, g, m, v in zip(ps, gs, ms, vs):
        g = g * coef
        p = p * (1 - lr * weight_decay)
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g * g
        p = p - (lr / bc1) * m / (v.sqrt() / bc2 ** 0.5 + eps)
        out_p.append(p), out_m.append(m), out_v.append(v)
    return out_p, out_m, out_v, total, coef


def adam_step_scale(m_scale, v, step, *, lr, betas, eps):
    """Magnitude of the Adam step lr / bc1 * m / (sqrt(v) / sqrt(bc2) + eps) with |m| replaced by `m_scale`, the sum of the
    magnitudes of the terms m is made of: where those terms cancel, the step is small but its rounding error is not."""
    b1, b2 = betas
    return lr / (1 - b1 ** step) * m_scale / (v.sqrt() / (1 - b2 ** step) ** 0.5 + eps)


def ulp32(x):
    """Spacing of fp32 numbers at |x| (float64 tensor on x's device)."""
    a = x.detach().to(torch.float32).abs()
    return (torch.nextafter(a, torch.full_like(a, float("inf"))) - a).double()


def graph_vs_eager(tr_graph, tr_eager, batches):
    """Runs `tr_graph` (cuda_graph=True) and `tr_eager` (same initial state) side by side over `batches`; the eager
    trainer is fed the noise and timesteps the graphed step drew. During capture those tensors are allocated in the
    graph's pool, so after every replay the references kept by the wrapped `add_noise` hold that replay's values.
    Returns per step (graphed loss, eager loss, graphed grad norm, eager grad norm), the drawn noises, and
    ||master_graph - master_eager|| / ||master_graph - master_initial|| after the last step."""
    drawn = {}
    real_add_noise = tr_graph.scheduler.add_noise

    def add_noise(original_samples, noise, timesteps):
        drawn["noise"], drawn["t"] = noise, timesteps
        return real_add_noise(original_samples, noise, timesteps)

    tr_graph.scheduler.add_noise = add_noise
    try:
        m0 = tr_graph.opt.master.clone()
        rows, noises = [], []
        for x in batches:
            la = float(tr_graph.step(x))
            noise, t = drawn["noise"].clone(), drawn["t"].clone()
            lb = float(tr_eager.step(x, noise=noise, timesteps=t))
            rows.append((la, lb, float(tr_graph.opt.grad_norm()), float(tr_eager.opt.grad_norm())))
            noises.append(noise)
        ma, mb = tr_graph.opt.master, tr_eager.opt.master
        drift = float((ma - mb).norm() / (ma - m0).norm().clamp_min(1e-30))
    finally:
        del tr_graph.scheduler.add_noise
    return rows, noises, drift
