"""The benchmarked workloads, kernel call by kernel call, at their own shapes.

bench.py times one LDMTrainer step of the 441 M-parameter U-Net (BASELINE config 3: 256/512/768 channels, batch 8 of
3 x 24^3 latents, bf16, every dispatch policy on `auto`) and the sampling forward of config 4 (32/64/128 channels on
1 x 1 x 128 x 128 x 64, attention at L = 32768). Tile sizes, split-K, the persistent tile loop, the upsample fold, the
GroupNorm statistics in the conv epilogue and the attention routing are all chosen from the shapes, so a test at a
smaller shape runs other code. Here every call the model makes to the ops entry points is recorded during one real
step and compared with an fp32 reference of the same operation on the same bf16 operands (TF32 off), per voxel and
per channel as well as globally: an error confined to one TMA box, one halo plane or one channel tile fails.

Bars (tests/callcheck.py, with the worst value observed on a B200 in the comment beside each):
  * one bf16 rounding of the result is off by at most 2^-8 = 3.9e-3 relative per element, 1.7e-3 rms on normally
    distributed values;
  * fp32 results (weight, bias and norm-gain gradients, the fp32 time-embedding path) only reorder fp32 sums;
  * attention stores P (forward) and dS (backward) in bf16 before the second product.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from callcheck import BARS, _attn_ref, _check_backward, _check_forward, _conv_ref, _peak, _Recorder, _Report
from util import BF16_TOL, assert_close_local, graph_vs_eager, local_errors, rel_err

DEV = "cuda"


@pytest.fixture
def no_tf32():
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


# ------------------------------------------------------------------------------------------------------------------
# the checker catches what rel_err misses (CPU)
# ------------------------------------------------------------------------------------------------------------------
def test_local_checker_catches_tile_faults():
    """On an 8 x 256 x 24^3 activation (level 0 of the benchmark): bf16 rounding noise passes; one 64-voxel box off by
    50 %, one channel off by 5 % and one boundary plane off by 10 % fail, and the message names the box / channel /
    plane -- while the global rel_err of all three stays under the 2e-2 bar the other parity tests use."""
    g = torch.Generator().manual_seed(0)
    want = torch.randn(8, 256, 24, 24, 24, generator=g)
    noise = want.to(torch.bfloat16).float()
    errs = assert_close_local(noise, want, what="bf16 rounding", **BARS["bf16"])
    assert errs["glob"] < 2e-3 and errs["row"] < 2.5e-3   # 1.66e-3 and 2.06e-3
    faults = {
        "box": (lambda t: t[5, :, 8:12, 4:8, 20:24].mul_(1.5), r"voxel \(n, \*spatial\) \(5, (8|9|10|11), [4-7], (2[0-3])\)"),
        "channel": (lambda t: t[:, 77].mul_(1.05), r"worst channel 77 "),
        "plane": (lambda t: t[3, :, :, :, 23].mul_(1.1), r"voxel \(n, \*spatial\) \(3, \d+, \d+, 23\)"),
    }
    for name, (inject, where) in faults.items():
        got = noise.clone()
        inject(got)
        assert rel_err(got, want) < BF16_TOL, name
        with pytest.raises(AssertionError, match=where):
            assert_close_local(got, want, what=name, **BARS["bf16"])


# ------------------------------------------------------------------------------------------------------------------
# the benchmark's models
# ------------------------------------------------------------------------------------------------------------------
def _bench_trainer(cuda_graph=True):
    """Model and trainer exactly as bench.run_b200 builds them."""
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import planner
    from medical_image_generation_b200.engine import LDMTrainer
    torch.manual_seed(0)
    model = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**bench.unet_kwargs(), compute_dtype=torch.bfloat16))
    model = model.to(DEV).train()
    sched = mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS)
    tr = LDMTrainer(model, sched, lr=2e-5, grad_clip_max_norm=1.0, cuda_graph=cuda_graph, bucket_mb=64.0,
                    graph_warmup_steps=2, shard_optimizer=None)
    return model, tr


def _bench_batch(seed, batch=8):
    import bench
    g = torch.Generator().manual_seed(seed)
    x0 = torch.randn((batch, *bench.LATENT), generator=g)
    noise = torch.randn(x0.shape, generator=g)
    t = torch.randint(0, 1000, (batch,), generator=g)
    return x0.to(DEV), noise.to(DEV), t.to(DEV)


@pytest.fixture(scope="module")
def bench_trainer():
    model, tr = _bench_trainer()
    yield model, tr
    tr.opt.close()
    del model, tr
    torch.cuda.empty_cache()


# C entry points one eager training step launches through ops (bench shape, defaults; recorded on a B200): the upsample
# fold at 12^3 -> 24^3 (mig_upconv_*, mig_class_interleave), the unfolded nearest upsample + conv at 6^3 -> 12^3 (too
# few tiles to fold), the unfused attention chain at 12^3 (d = 512: mig_gemm_strided, mig_softmax_fwd,
# mig_softmax_bwd_narrow), flash at 6^3 (d = 768, L = 216) and the GroupNorm statistics in the conv epilogue
# (mig_conv_fwd_stats, mig_groupnorm_apply). A routing change that moves the benchmark onto another path fails here:
# make sure the new path is among the calls checked in this file, then update the list.
TRAIN_STEP_CALLS = sorted([
    "mig_add", "mig_class_interleave", "mig_colsum", "mig_concat_channels", "mig_conv_dgrad", "mig_conv_fwd",
    "mig_conv_fwd_stats", "mig_conv_wgrad", "mig_flash_attention_bwd", "mig_flash_attention_fwd_ld",
    "mig_gemm_strided", "mig_groupnorm_apply", "mig_groupnorm_bwd", "mig_groupnorm_fwd", "mig_mse_bwd", "mig_mse_fwd",
    "mig_nchw_to_nhwc", "mig_nhwc_to_nchw", "mig_silu_bwd", "mig_silu_fwd", "mig_softmax_bwd_narrow",
    "mig_softmax_fwd", "mig_split_channels", "mig_temb_proj_all_bwd", "mig_temb_proj_all_fwd", "mig_timestep_embedding",
    "mig_upconv_fold_filter", "mig_upconv_fwd", "mig_upconv_unfold_wgrad", "mig_upsample_nearest_bwd",
    "mig_upsample_nearest_fwd",
])

# ... and of one config-4 sampling forward: both upsample convs folded, flash at L = 32768, the filters cast to bf16
# once (mig_cast: no optimiser keeps a shadow), the one-channel input already channels-last.
SAMPLING_CALLS = sorted([
    "mig_add", "mig_cast", "mig_concat_channels", "mig_conv_fwd", "mig_conv_fwd_stats", "mig_flash_attention_fwd_ld",
    "mig_groupnorm_apply", "mig_groupnorm_fwd", "mig_nhwc_to_nchw", "mig_silu_fwd", "mig_temb_proj_all_fwd",
    "mig_timestep_embedding", "mig_upconv_fold_filter", "mig_upconv_fwd",
])


@pytest.mark.gpu
def test_training_step_calls_at_bench_shape(bench_trainer, monkeypatch, no_tf32):
    """Every distinct ops call of one eager LDMTrainer step at the benchmark shape: forward in place, backward
    standalone, plus the epilogue GroupNorm statistics, the bf16 shadow and the C entry points the step used."""
    from medical_image_generation_b200 import ops
    model, tr = bench_trainer
    torch.cuda.reset_peak_memory_stats()
    rep = _Report("training step, BASELINE config 3")
    recorder = _Recorder(monkeypatch, ops)
    x0, noise, t = _bench_batch(1000)
    tr._eager_step(x0, noise, t)
    torch.cuda.synchronize()
    recorder.on = False
    rep.require(recorder.names == set(TRAIN_STEP_CALLS), f"entry points: {sorted(recorder.names)} (expected "
                f"{TRAIN_STEP_CALLS}; missing {sorted(set(TRAIN_STEP_CALLS) - recorder.names)}, new "
                f"{sorted(recorder.names - set(TRAIN_STEP_CALLS))})")
    # the bf16 filters every tensor-core kernel reads are the round-to-nearest of the fp32 masters, bit for bit
    rep.require(torch.equal(tr.opt.shadow, tr.opt.master.to(torch.bfloat16)), "bf16 shadow != bf16(master)")
    ops_seen = {}
    for rec in recorder.calls.values():
        ops_seen[rec["op"]] = ops_seen.get(rec["op"], 0) + 1
        _check_forward(rep, rec)
        _check_backward(rep, recorder.real, rec)
    rep.require({"conv", "upconv", "gn", "linear", "temb", "sdpa_qkv"} <= set(ops_seen), f"ops recorded: {ops_seen}")
    rep.require(any(r["op"] == "conv" and r["sums"] is not None for r in recorder.calls.values()),
                "no conv delivered epilogue GroupNorm statistics")
    rep.require(any(r["op"] == "upconv" and r["sig"][-1] for r in recorder.calls.values()), "the upsample fold did not run")
    print(f"distinct calls checked: {ops_seen}")
    _peak(rep, "training calls")
    rep.finish()


@pytest.mark.gpu
def test_sampling_forward_calls_at_bench_shape(monkeypatch, no_tf32):
    """Every distinct ops call of one config-4 sampling forward (1 x 1 x 128 x 128 x 64, no_grad): the 32-channel
    halo kernels at a million voxels, the narrow tiles with epilogue statistics and flash attention at L = 32768."""
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import ops
    torch.cuda.reset_peak_memory_stats()
    torch.manual_seed(7)
    model = bench.rerandomize_zero_init(mig.DiffusionModelUNet(**bench.SAMPLING_CFG, compute_dtype=torch.bfloat16))
    model = model.to(DEV).eval()
    x = torch.randn((1, *bench.VOLUME), generator=torch.Generator().manual_seed(42)).to(DEV)
    rep = _Report("sampling forward, BASELINE config 4")
    recorder = _Recorder(monkeypatch, ops)
    with torch.no_grad():
        model(x, torch.tensor([500], device=DEV))
    torch.cuda.synchronize()
    recorder.on = False
    rep.require(recorder.names == set(SAMPLING_CALLS), f"entry points: {sorted(recorder.names)} (expected {SAMPLING_CALLS})")
    attn = [r for r in recorder.calls.values() if r["op"] == "sdpa_qkv"]
    rep.require([r["qkv"].shape[1] for r in attn] == [32768], f"attention lengths {[r['qkv'].shape for r in attn]}")
    for rec in recorder.calls.values():
        _check_forward(rep, rec)
    _peak(rep, "sampling calls")
    rep.finish()


# ------------------------------------------------------------------------------------------------------------------
# attention at the lengths the benchmarks use
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,L,C", [(1, 8192, 128), (1, 32768, 128)])
def test_flash_attention_at_sampling_lengths(B, L, C, monkeypatch, no_tf32):
    """Fused forward and backward at L = 8192 and 32768 (64 / 256 KV blocks per query tile), checked per query row."""
    from medical_image_generation_b200 import ops
    g = torch.Generator().manual_seed(L)
    q, k, v, dO = (torch.randn(B, L, C, generator=g).to(DEV, torch.bfloat16) for _ in range(4))
    scale = 1 / math.sqrt(C)
    seen = []
    real = ops.call
    monkeypatch.setattr(ops, "call", lambda name, *a: (seen.append(name), real(name, *a))[1])
    qd, kd, vd = (t.clone().requires_grad_(True) for t in (q, k, v))
    out = ops.sdpa(qd, kd, vd, 1, scale)
    out.backward(dO)
    monkeypatch.setattr(ops, "call", real)
    rep = _Report(f"flash attention B={B} L={L} C={C}")
    rep.require(seen == ["mig_flash_attention_fwd_ld", "mig_flash_attention_bwd"], f"calls {seen}")
    qr, kr, vr = (t.float().requires_grad_(True) for t in (q, k, v))
    want = _attn_ref(qr, kr, vr, 1, scale)
    want.backward(dO.float())
    for name, got, ref in (("out", out, want), ("dq", qd.grad, qr.grad), ("dk", kd.grad, kr.grad), ("dv", vd.grad, vr.grad)):
        rep.local("attn", got, ref, f"flash L={L} {name}")
    rep.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,C,path", [(8, 1728, 512, "unfused"), (8, 216, 768, "flash")])
def test_sdpa_qkv_routing_at_training_shapes(B, L, C, path, monkeypatch, no_tf32):
    """The two attention blocks of the training step in `auto`: d = 512 at L = 1728 takes the unfused GEMM + softmax
    chain (row stride 3C, dS narrowed to bf16), d = 768 at L = 216 the fused kernels; order as the flat optimiser lays
    out the projections."""
    from medical_image_generation_b200 import ops
    order = ("v", "k", "q")
    g = torch.Generator().manual_seed(L + C)
    qkv = torch.randn(B, L, 3 * C, generator=g).to(DEV, torch.bfloat16)
    dO = torch.randn(B, L, C, generator=g).to(DEV, torch.bfloat16)
    scale = 1 / math.sqrt(C)
    seen = set()
    real = ops.call
    monkeypatch.setattr(ops, "call", lambda name, *a: (seen.add(name), real(name, *a))[1])
    qd = qkv.clone().requires_grad_(True)
    out = ops.sdpa_qkv(qd, 1, scale, order)
    out.backward(dO)
    monkeypatch.setattr(ops, "call", real)
    expected = ({"mig_gemm_strided", "mig_softmax_fwd", "mig_softmax_bwd_narrow"} if path == "unfused" else
                {"mig_flash_attention_fwd_ld", "mig_flash_attention_bwd", "mig_concat_channels"})
    rep = _Report(f"sdpa_qkv B={B} L={L} C={C}")
    rep.require(seen == expected, f"calls {sorted(seen)}, expected {sorted(expected)}")
    qr = qkv.float().requires_grad_(True)
    sl = {n: qr[..., i * C:(i + 1) * C] for i, n in enumerate(order)}
    want = _attn_ref(sl["q"], sl["k"], sl["v"], 1, scale)
    want.backward(dO.float())
    rep.local("attn", out, want, f"sdpa_qkv {path} out")
    rep.local("attn", qd.grad, qr.grad, f"sdpa_qkv {path} dqkv")
    rep.finish()


@pytest.mark.gpu
def test_fp32_reference_matches_fp64(no_tf32):
    """The references above run in fp32 on the GPU with TF32 off; on bf16 operands they agree with fp64 on the CPU."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 64, 6, 6, 6, generator=g).bfloat16().float()
    w = (torch.randn(96, 64, 3, 3, 3, generator=g) / 40).bfloat16().float()
    b, cb = torch.randn(96, generator=g), torch.randn(2, 96, generator=g)
    want = _conv_ref(x.double(), w.double(), b.double(), (1, 1, 1), (1, 1, 1), cb.double())
    got = _conv_ref(x.to(DEV), w.to(DEV), b.to(DEV), (1, 1, 1), (1, 1, 1), cb.to(DEV))
    assert rel_err(got, want) < 1e-6
    gn = F.silu(F.group_norm(x.to(DEV), 32, b[:64].to(DEV), cb[0, :64].to(DEV), 1e-6))
    assert rel_err(gn, F.silu(F.group_norm(x.double(), 32, b[:64].double(), cb[0, :64].double(), 1e-6))) < 1e-6
    q, k, v = (torch.randn(2, 216, 256, generator=g).bfloat16().float() for _ in range(3))
    got = _attn_ref(q.to(DEV), k.to(DEV), v.to(DEV), 2, 1 / 16, rows=100)
    assert rel_err(got, _attn_ref(q.double(), k.double(), v.double(), 2, 1 / 16)) < 1e-6


# ------------------------------------------------------------------------------------------------------------------
# the whole step against the oracle, and the graph replay against eager steps
# ------------------------------------------------------------------------------------------------------------------
# whole step against the oracle (the golden model tests use 2e-2 output, 8e-2 gradient)
OUT_BAR = 1e-2       # worst 3.7e-3
GRAD_BAR = 6e-2      # worst 3.1e-2 (up_blocks.1.attentions.1.to_q.bias)
LOSS_BAR = 5e-3      # worst 5.2e-4
NORM_BAR = 5e-3      # worst 6.4e-4

# graphed vs eager steps on the same inputs: GroupNorm / split-K atomics reorder fp32 sums between the two runs
GRAPH_LOSS_BAR = 2e-3    # worst 1.3e-4
GRAPH_NORM_BAR = 5e-3    # worst 8.1e-4
GRAPH_DRIFT_BAR = 0.2    # worst 3.7e-2; a stale input, noise or shadow gives about 1


@pytest.mark.gpu
def test_training_step_matches_oracle_at_bench_shape(bench_trainer, monkeypatch, no_tf32):
    """One production step (batch 8) and the fp32 oracle (plain torch, pinned to the reference goldens) on the same
    weights and batch: loss, U-Net output, every parameter's full gradient and the global gradient norm."""
    import bench
    from oracle import torch_oracle as O
    model, tr = bench_trainer
    torch.cuda.reset_peak_memory_stats()
    cfg = bench.unet_kwargs()
    params = {k: v.detach().float().contiguous().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    x0, noise, t = _bench_batch(2000)
    got = {}
    hook = model.register_forward_hook(lambda m, a, kw, out: got.update(x=kw["x"].detach().clone(), out=out.detach().clone()),
                                       with_kwargs=True)
    try:
        loss = float(tr._eager_step(x0, noise, t).detach())
    finally:
        hook.remove()
    real_temb = O.timestep_embedding    # (builds its frequency table on the CPU)
    monkeypatch.setattr(O, "timestep_embedding", lambda ts, dim, max_period=10000: real_temb(ts.cpu(), dim, max_period).to(ts.device))
    pred = O.unet_forward(params, cfg, got["x"], t)
    ref_loss = F.mse_loss(pred, noise)
    ref_loss.backward()
    rep = _Report("training step vs oracle, BASELINE config 3")
    rep.value("loss", abs(loss - float(ref_loss)) / float(ref_loss), LOSS_BAR, "loss")
    rep.value("output", rel_err(got["out"], pred), OUT_BAR, "U-Net output (rel_err)")
    e = local_errors(got["out"], pred)
    print(f"U-Net output: per-voxel {e['row']:.3e} at {e['row_at']}, per-channel {e['col']:.3e}")
    named = dict(model.named_parameters())
    sq = 0.0
    for k, p in named.items():
        ref = params[k].grad
        if ref is None:
            rep.require("proj_attn" in k, f"oracle gives no gradient for {k}")
            continue
        sq += float(ref.double().pow(2).sum())
        if k.endswith("to_k.bias"):
            continue    # exactly zero mathematically (softmax is shift invariant): noise on both sides
        rep.value("param grad", rel_err(p.main_grad, ref, floor=1e-12), GRAD_BAR, k)
    rep.value("grad_norm", abs(float(tr.opt.grad_norm()) - sq ** 0.5) / sq ** 0.5, NORM_BAR, "opt.grad_norm()")
    _peak(rep, "oracle step")
    rep.finish()


@pytest.mark.gpu
def test_graph_replay_matches_eager_at_bench_shape():
    """Capture and three replays of the benchmarked CUDA-graph step against eager steps of a second trainer fed the
    same batch, noise and timesteps: a replay that reads a stale input, noise or shadow weights moves the masters
    elsewhere (drift ratio near 1)."""
    torch.cuda.reset_peak_memory_stats()
    model_a, tr_a = _bench_trainer(cuda_graph=True)
    import bench
    import medical_image_generation_b200 as mig
    from medical_image_generation_b200 import planner
    from medical_image_generation_b200.engine import LDMTrainer
    model_b = mig.DiffusionModelUNet(**bench.unet_kwargs(), compute_dtype=torch.bfloat16)
    model_b.load_state_dict(model_a.state_dict())
    tr_b = LDMTrainer(model_b.to(DEV).train(), mig.DDPMScheduler(**planner.LDM_SCHEDULER_KWARGS), lr=2e-5,
                      grad_clip_max_norm=1.0)
    batches = [_bench_batch(3000 + i)[0] for i in range(6)]
    rows, noises, drift = graph_vs_eager(tr_a, tr_b, batches)
    rep = _Report("graph replay vs eager, BASELINE config 3")
    rep.require(tr_a._graph is not None and int(tr_a.opt.step_dev) == 6, "capture did not happen")
    rep.require(not any(torch.equal(noises[i], noises[i + 1]) for i in range(2, 5)), "replays drew the same noise")
    for i, (la, lb, ga, gb) in enumerate(rows):
        rep.value("loss", abs(la - lb) / abs(lb), GRAPH_LOSS_BAR, f"step {i} loss {la:.5f} vs {lb:.5f}")
        rep.value("grad_norm", abs(ga - gb) / gb, GRAPH_NORM_BAR, f"step {i} grad norm {ga:.5f} vs {gb:.5f}")
    rep.value("master drift", drift, GRAPH_DRIFT_BAR, "||master_A - master_B|| / ||master_A - master_0||")
    _peak(rep, "two trainers")
    tr_a.opt.close()
    tr_b.opt.close()
    del tr_a, tr_b, model_a, model_b
    torch.cuda.empty_cache()
    rep.finish()
