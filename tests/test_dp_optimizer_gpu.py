"""FlatAdamW across data-parallel ranks with gradients injected straight into `main_grad`, so no U-Net and none of its
nondeterminism is in the comparison. On every rank a sharded optimiser (`shard=True`: reduce-scatter, the strided kernels
on the owned slices, all-gather of the bf16 shadow) and a replicated one (`shard=False`: all-reduce, one contiguous
step) update identical copies of a small module with the same gradients. The mean gradient of two ranks is the same
bits under both schemes, so with the clip inactive the two must agree bit for bit; with it active only the rounding of
the partial sums of ||g||^2 differs. Both are also checked per element against the fp64 reference.

gloo at world 2 with both ranks on cuda:0 always runs (it takes ShardedBuckets' all_reduce + divide and list all_gather
branches); NCCL, one rank per GPU, runs the production branches (reduce_scatter_tensor(AVG), the coalesced gather) and
the CUDA-graph replay of the sharded LDM step when at least two GPUs are visible."""
import copy
import os
import random
import socket
from datetime import timedelta

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

from util import adam_step_scale, clip_adamw_reference, f32, ulp32

pytestmark = pytest.mark.gpu

HP = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2)
BUCKET_MB = 1536 * 4 / (1 << 20)   # 1536-element buckets: 4 of them at W = 2, 4, 8 (3 at W = 5, 7)
STEPS = 4
SCALES = {"clip_inactive": 1e-3, "clip_active": 1.0}   # gradient element scale: ||g|| about 0.1 and 100, max_norm 1

# bars, with the worst value measured on a B200 next to each
NORM_TOL = 5e-7        # grad_norm() against the fp64 norm of the mean gradient, relative; 6.2e-8
REF_M_TOL = 1.5e-6     # after STEPS steps: |m - m_ref| / m_scale (m_scale: the same recurrence over |clip g|); 3.0e-7
REF_V_TOL = 2e-6       # |v - v_ref| / v_ref; 4.5e-7
REF_P_ULP, REF_P_REL = 2.0 * STEPS, 1e-6   # |p - p_ref| <= REF_P_ULP ulp(p_ref) + REF_P_REL p_scale, where p_scale sums
#                                            |weight decay| + |Adam step| (util.adam_step_scale) over the steps; beyond
#                                            the ulp term: 1.3e-7
CLIP_TOL = 2e-6        # sharded against replicated with the clip active, on the same scales as the REF_ bars; m 1.8e-7,
#                        v 4.2e-7, p beyond the ulp term 1.0e-7 (gloo, world 2)


class Toy(nn.Module):
    """Weights whose sizes are not multiples of 64 (one channels-last conv filter), 1-D biases, a `time_embed` Linear
    (fp32-consumed: replicated region) and a `proj_attn` Linear (never gets a gradient: unused tail). In buffer order the
    sharded members are 1344 / 2496 / 192 / 512 / 256 padded elements: with 1536-element buckets the conv filter spans
    three buckets and bucket 2 holds four members."""

    def __init__(self):
        super().__init__()
        self.conv_a = nn.Conv3d(7, 13, 3)
        self.conv_a.weight.data = self.conv_a.weight.data.contiguous(memory_format=torch.channels_last_3d)
        self.lin_b = nn.Linear(29, 45)
        self.w_c = nn.Parameter(torch.randn(70, 3))
        self.w_d = nn.Parameter(torch.randn(9, 8, 7))
        self.w_e = nn.Parameter(torch.randn(33, 5))
        self.time_embed = nn.Linear(24, 40)
        self.proj_attn = nn.Linear(16, 16)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _init(rank, world, port, backend):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", 0 if backend == "gloo" else rank)
    torch.cuda.set_device(dev)
    kw = dict(device_id=dev) if backend == "nccl" else {}
    dist.init_process_group(backend, rank=rank, world_size=world, timeout=timedelta(seconds=120), **kw)
    return dev


def _spawn(fn, world, *args):
    from medical_image_generation_b200 import _lib
    _lib.load()     # fail here, not in every rank, when the library is missing
    mp.spawn(fn, args=(world, _free_port(), *args), nprocs=world, join=True)


def _grads(trained, step, rank, micro, scale):
    gen = torch.Generator().manual_seed(1_000_003 * step + 1009 * rank + micro)
    return [torch.randn(p.shape, generator=gen) * scale for _, p in trained]


def _same_on_all_ranks(t):
    bits = t.contiguous().view(torch.int32)
    parts = [torch.empty_like(bits) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, bits)
    return all(torch.equal(q, bits) for q in parts)


def _slot(opt, buf, p):
    off, k = p._mig_slot
    return buf[off:off + k].as_strided(p.shape, p.stride())


def _check_shadow(opt):
    """bf16 shadow == bf16(master) wherever this rank's master is current: the owned slices and the replicated region
    (sharded), the whole buffer (replicated)."""
    if opt.sharded:
        bk = opt.buckets
        ok = all(torch.equal(bk.owned(opt.shadow, b), bk.owned(opt.master, b).to(torch.bfloat16)) for b in range(bk.nb))
        lo = opt.repl_lo
        return ok and torch.equal(opt.shadow[lo:], opt.master[lo:].to(torch.bfloat16))
    return torch.equal(opt.shadow, opt.master.to(torch.bfloat16))


def _worker(rank, world, port, backend):
    dev = _init(rank, world, port, backend)
    try:
        from medical_image_generation_b200.engine import FlatAdamW
        exact = backend == "gloo" or world == 2     # (a + b) / 2 has one rounding whatever the collective
        hp32 = dict(lr=f32(HP["lr"]), betas=tuple(f32(b) for b in HP["betas"]), eps=f32(HP["eps"]),
                    weight_decay=f32(HP["weight_decay"]))
        for case, scale in SCALES.items():
            for accumulate in (False, True):
                torch.manual_seed(0)
                base = Toy().to(dev)
                mods = {"sharded": base, "replicated": copy.deepcopy(base)}
                init = {n: p.detach().clone() for n, p in base.named_parameters()}
                opts = {k: FlatAdamW(m, max_grad_norm=1.0, bucket_mb=BUCKET_MB, shard=(k == "sharded"), **HP)
                        for k, m in mods.items()}
                sh, rep = opts["sharded"], opts["replicated"]
                assert sh.sharded and not rep.sharded
                bk = sh.buckets
                assert bk.nb >= 3 and any(len(b) >= 2 for b in bk.member_buckets)
                assert max(b["n"] for b in bk.buckets[:bk.nb]) >= 3
                trained = {k: [(n, p) for n, p in m.named_parameters() if "proj_attn" not in n] for k, m in mods.items()}
                ref_p = [init[n].double() for n, _ in trained["sharded"]]
                ref_m = [torch.zeros_like(q) for q in ref_p]
                ref_v = [torch.zeros_like(q) for q in ref_p]
                m_scale = [torch.zeros_like(q) for q in ref_p]
                p_move = [torch.zeros_like(q) for q in ref_p]
                micros = (0, 1) if accumulate else (0,)
                for step in range(1, STEPS + 1):
                    for opt in opts.values():
                        opt.zero_grad()
                    order = list(range(len(trained["sharded"])))
                    for micro in micros:
                        random.Random(step * 10 + micro).shuffle(order)   # same order on every rank, like backward
                        last = micro == micros[-1]
                        for k, opt in opts.items():
                            opt.set_grad_sync(last)
                            for (_, p), gr in zip(trained[k], _grads(trained[k], step, rank, micro, scale)):
                                p.main_grad.add_(gr.to(dev))
                            for i in order:
                                p = trained[k][i][1]
                                p._mig_grad_ready(p)
                    for opt in opts.values():
                        opt.step()
                    # fp64 reference on the mean gradient of all ranks
                    mean = [torch.zeros_like(q) for q in ref_p]
                    for r in range(world):
                        for micro in micros:
                            for acc, gr in zip(mean, _grads(trained["sharded"], step, r, micro, scale)):
                                acc += gr.to(dev).double() / world
                    ref_p0 = ref_p
                    ref_p, ref_m, ref_v, total, coef = clip_adamw_reference(ref_p, mean, ref_m, ref_v, step,
                                                                            max_norm=1.0, **hp32)
                    m_scale = [hp32["betas"][0] * s + (1 - hp32["betas"][0]) * (g * coef).abs()
                               for s, g in zip(m_scale, mean)]
                    p_move = [mv + (q * hp32["lr"] * hp32["weight_decay"]).abs() +
                              adam_step_scale(s, v, step, lr=hp32["lr"], betas=hp32["betas"], eps=hp32["eps"])
                              for mv, q, s, v in zip(p_move, ref_p0, m_scale, ref_v)]
                    for k, opt in opts.items():
                        gn = float(opt.grad_norm())
                        err = abs(gn - float(total)) / float(total)
                        print(f"measured {backend} W={world} {case} acc={accumulate} step {step} {k} "
                              f"grad_norm rel err: {err:.3e}")
                        assert err <= NORM_TOL, (k, step, gn, float(total))
                        assert _same_on_all_ranks(opt.shadow), f"{k}: bf16 shadows differ across ranks"
                        assert _check_shadow(opt), f"{k}: shadow != bf16(master)"
                    if case == "clip_inactive" and exact:   # (the layouts differ: compare parameter by parameter)
                        for (n, pa), (_, pb) in zip(mods["sharded"].named_parameters(), mods["replicated"].named_parameters()):
                            assert torch.equal(pa._mig_shadow, pb._mig_shadow), f"gathered shadow of {n} != replicated"
                sh.consolidate()
                rep.consolidate()
                for opt in opts.values():
                    for buf in (opt.master, opt.m, opt.v):
                        assert _same_on_all_ranks(buf), "master / moments differ across ranks after consolidate()"
                    assert _check_shadow(opt)
                for n, p in mods["sharded"].named_parameters():
                    if "proj_attn" in n:
                        assert torch.equal(p.detach(), init[n]), "an unused parameter moved"
                if case == "clip_inactive" and exact:
                    for (n, pa), (_, pb) in zip(trained["sharded"], trained["replicated"]):
                        assert torch.equal(pa.detach(), pb.detach()), f"sharded {n} != replicated"
                        for buf in ("m", "v"):
                            assert torch.equal(_slot(sh, getattr(sh, buf), pa), _slot(rep, getattr(rep, buf), pb)), \
                                f"sharded {buf} of {n} != replicated"
                sa, sb = sh.torch_state_dict(), rep.torch_state_dict()
                assert sorted(sa["state"]) == sorted(sb["state"]) and sa["param_groups"] == sb["param_groups"]
                for i, st in sa["state"].items():
                    assert float(st["step"]) == float(sb["state"][i]["step"]) == STEPS
                    if case == "clip_inactive" and exact:
                        for key in ("exp_avg", "exp_avg_sq"):
                            assert torch.equal(st[key], sb["state"][i][key]), ("torch_state_dict", i, key)
                worst = {}
                for j, ((n, pa), (_, pb)) in enumerate(zip(trained["sharded"], trained["replicated"])):
                    pr, mr, vr, ms, mv = ref_p[j], ref_m[j], ref_v[j], m_scale[j], p_move[j]
                    ulp = ulp32(pr)
                    for k, opt, p in (("sharded", sh, pa), ("replicated", rep, pb)):
                        em = (_slot(opt, opt.m, p).double() - mr).abs() / ms.clamp_min(1e-300)
                        ev = (_slot(opt, opt.v, p).double() - vr).abs() / vr.clamp_min(1e-300)
                        ep = (p.detach().double() - pr).abs()
                        worst[k + " m"] = max(worst.get(k + " m", 0.0), float(em.max()))
                        worst[k + " v"] = max(worst.get(k + " v", 0.0), float(ev.max()))
                        beyond = (ep - REF_P_ULP * ulp).clamp_min(0) / mv
                        worst[k + " p beyond ulp"] = max(worst.get(k + " p beyond ulp", 0.0), float(beyond.max()))
                        assert bool((em <= REF_M_TOL).all()) and bool((ev <= REF_V_TOL).all()), (k, n)
                        assert bool((ep <= REF_P_ULP * ulp + REF_P_REL * mv).all()), (k, n, float((ep / ulp).max()))
                    dm = (_slot(sh, sh.m, pa) - _slot(rep, rep.m, pb)).double().abs() / ms.clamp_min(1e-300)
                    dv = (_slot(sh, sh.v, pa) - _slot(rep, rep.v, pb)).double().abs() / vr.clamp_min(1e-300)
                    dp = (pa.detach() - pb.detach()).double().abs()
                    beyond = (dp - REF_P_ULP * ulp).clamp_min(0) / mv
                    worst["sharded-replicated p beyond ulp"] = max(worst.get("sharded-replicated p beyond ulp", 0.0),
                                                                   float(beyond.max()))
                    worst["sharded-replicated m"] = max(worst.get("sharded-replicated m", 0.0), float(dm.max()))
                    worst["sharded-replicated v"] = max(worst.get("sharded-replicated v", 0.0), float(dv.max()))
                    assert bool((dm <= CLIP_TOL).all()) and bool((dv <= CLIP_TOL).all()), n
                    assert bool((dp <= REF_P_ULP * ulp + CLIP_TOL * mv).all()), n
                print(f"measured {backend} W={world} {case} acc={accumulate}: " +
                      ", ".join(f"{k} {v:.3e}" for k, v in worst.items()))
                for opt in opts.values():
                    opt.close()
    finally:
        dist.destroy_process_group()


def test_flat_adamw_sharded_matches_replicated_gloo_world2():
    """gloo, world 2, both ranks on cuda:0."""
    _spawn(_worker, 2, "gloo")


def _gpus_or_skip():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"NCCL data parallel needs at least 2 visible GPUs, {n} visible")
    return n


def test_flat_adamw_sharded_matches_replicated_nccl():
    """NCCL, one rank per GPU, world = min(8, visible GPUs). For W > 2 the AVG reductions may round differently from
    the all-reduce, so sharded and replicated are held to the clip-active bar instead of bit equality."""
    _spawn(_worker, min(8, _gpus_or_skip()), "nccl")


def _graph_worker(rank, world, port):
    dev = _init(rank, world, port, "nccl")
    try:
        import medical_image_generation_b200 as mig
        from medical_image_generation_b200.engine import LDMTrainer
        from oracle.golden_util import golden_params
        from test_models_gpu import GRAPH_DRIFT_TOL, GRAPH_LOSS_TOL, GRAPH_NORM_TOL
        from util import graph_vs_eager
        g = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "unet3d_small.pt"),
                       weights_only=False)
        params = golden_params(g["shapes"], g["seed"])
        kw = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0015, beta_end=0.0205)
        trainers = []
        for graph in (True, False):
            m = mig.DiffusionModelUNet(**g["cfg"], compute_dtype=torch.bfloat16)
            m.load_state_dict(params)
            trainers.append(LDMTrainer(m.to(dev).train(), mig.DDPMScheduler(**kw), lr=1e-4, cuda_graph=graph,
                                       graph_warmup_steps=2, bucket_mb=0.25))
        tr, tr_eager = trainers
        assert tr.opt.sharded and tr_eager.opt.sharded and tr.opt.buckets.nb > 1
        gen = torch.Generator().manual_seed(4 + rank)
        xs = [torch.randn(2, 3, 8, 8, 8, generator=gen).to(dev) for _ in range(7)]
        rows, noises, drift = graph_vs_eager(tr, tr_eager, xs)
        assert tr._graph is not None, "capture did not happen"
        assert int(tr.opt.step_dev) == 7 and tr.opt.step_count == 7
        for la, lb, ga, gb in rows:
            assert abs(la - lb) < GRAPH_LOSS_TOL * abs(lb) and abs(ga - gb) < GRAPH_NORM_TOL * gb, rows
        assert drift < GRAPH_DRIFT_TOL, drift
        for t in trainers:
            assert _same_on_all_ranks(t.opt.shadow), "bf16 shadows differ across ranks"
            t.opt.consolidate()
            assert _same_on_all_ranks(t.opt.master) and _check_shadow(t.opt)
            t.opt.close()
    finally:
        dist.destroy_process_group()


def test_sharded_cuda_graph_replay_nccl_world2():
    """The configuration bench.py trains at more than one GPU: LDMTrainer(cuda_graph=True) with the sharded optimiser,
    every replay against an eager sharded trainer fed the same noise and timesteps (small bf16 U-Net, several buckets)."""
    _gpus_or_skip()
    _spawn(_graph_worker, 2)
