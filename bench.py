#!/usr/bin/env python
"""Benchmark of the VTMAE train step (BASELINE.json metric: train samples/sec, fwd+bwd+AdamW).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): the canonical train.py model (64x64x12 image frame-stack +
two 32x32x12 tactile maps, dim 256, enc 4x / dec 3x, mask 0.95, early_conv_masking=False),
batch 256 per GPU, bf16 tensor-core compute with fp32 master weights / accumulation, synthetic
data, random-init weights.  One "step" = zero_grad + forward + backward (+ gradient all-reduce for
N > 1) + clip_grad_norm_(0.5) + AdamW, i.e. the reference's models/pretrain_models.py:707-711.

`--dump-outputs DIR` writes, after the K timed steps, what the last of them handed back to its caller
(see dump_outputs) as DIR/<name>.npy.  Weights and inputs are seeded, so the same arguments give the same
inputs on every run and two builds of the project can be compared output for output.

Prints ONE JSON line on rank 0.  `value` = whole-job samples/s with inputs resident in HBM;
`e2e` = the same metric through the public module API with pinned HOST inputs (H2D copy of every
step's batch and a D2H read of the loss inside the timed region).  `--impl reference` times the
reference algorithm's CPU path (the oracle port of the reference's PyTorch code; the reference tree
itself does not exist on the GPU box) on the host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

FLOPS_PER_SAMPLE = 3404.7e6  # fwd + bwd, SURVEY.md §8(d) / BASELINE.md §3 (sum of 2*M*N*K, x3)
BATCH_PER_GPU = 256
WORKLOAD = "VTMAE pretrain step, canonical train.py model, batch 256/GPU, bf16 (BASELINE.json configs[1])"


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
                self.lines = [l for l in out.splitlines() if l.strip()]
            except Exception:
                self.proc.kill()
        return False

    def summary(self):
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def build_model(device):
    import torch
    from m3l_b200 import VTT, VTMAE
    torch.manual_seed(0)
    enc = VTT(image_size=(64, 64), tactile_size=(32, 32), image_patch_size=8, tactile_patch_size=4, dim=256, depth=4,
              heads=4, mlp_dim=512, num_tactiles=2, image_channels=12, tactile_channels=12, frame_stack=4)
    mae = VTMAE(encoder=enc, decoder_dim=256, masking_ratio=0.95, decoder_depth=3, decoder_heads=4, num_tactiles=2,
                early_conv_masking=False, frame_stack=4)
    return mae.to(device)


def synth_obs(B, seed, pinned=True, u8_frames=False):
    """One rollout-buffer batch as the reference's learners hold it (ppo_mae.py:236-262): image frames
    [B, F, 64, 64, 3] in [0, 1] and tactile maps [B, F, 6, 32, 32] in [-1, 1], fp32 (u8_frames: the compact storage
    variant, uint8 frames scaled by 1/255 on the device), plus the mask noise."""
    import torch
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(B, 4, 64, 64, 3, generator=g)
    if u8_frames:
        img = (img * 255).to(torch.uint8)
    obs = {"image": img, "tactile": torch.rand(B, 4, 6, 32, 32, generator=g) * 2 - 1}
    noise = torch.rand(B, 192, generator=g)
    if pinned:
        obs = {k: v.pin_memory() for k, v in obs.items()}
        noise = noise.pin_memory()
    return obs, noise


def synth_batch(B, seed, pinned=False):
    import torch
    g = torch.Generator().manual_seed(seed)
    x = {"image": torch.rand(B, 12, 64, 64, generator=g), "tactile1": torch.rand(B, 12, 32, 32, generator=g),
         "tactile2": torch.rand(B, 12, 32, 32, generator=g)}
    noise = torch.rand(B, 192, generator=g)
    if pinned:
        x = {k: v.pin_memory() for k, v in x.items()}
        noise = noise.pin_memory()
    return x, noise


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(steps: int, warmup: int, batch: int = 32):
    """Times zero_grad+fwd+bwd+clip+AdamW of the oracle (port of the reference's PyTorch code) in fp32
    on all host cores, on a `batch`-sample slice of the workload.  Returns (samples/s, ms/step, cores)."""
    import torch
    from oracle import vtmae_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = O.VTMAEConfig()
    sd = O.init_state_dict(cfg, seed=0)
    x, _ = synth_batch(batch, 1234)
    g = torch.Generator().manual_seed(1)
    noise = O.tie_free_noise(batch, 192, g, [64, 64, 64])
    st = O.AdamWState()
    for _ in range(warmup):
        O.train_step(sd, cfg, x, noise, st)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.train_step(sd, cfg, x, noise, st)
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps * 1e3, cores


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    sps, ms, cores = cpu_reference_run(steps, max(1, min(args.warmup, 3)))
    sample = f"batch 32 slice of the 256/GPU workload, fp32, torch CPU, {cores} threads, {steps} timed steps"
    line = {"impl": "reference", "metric": "VTMAE train samples/sec (fwd+bwd+AdamW)", "value": sps, "unit": "samples/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": sample},
            "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def time_kernel(fn, iters=10):
    import torch
    for _ in range(2):
        fn()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters * 1e-3  # seconds


def _flush_l2():
    import torch
    global _FLUSH
    try:
        _FLUSH.zero_()
    except NameError:
        _FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        _FLUSH.zero_()


def time_kernel_cold(fn, iters=8):
    """Median CUDA-event time of one launch with the L2 flushed (256 MB write) before every launch."""
    import torch
    for _ in range(2):
        fn()
    ts = []
    for _ in range(iters):
        _flush_l2()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2]


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures
# (profiles/r02_ncu_top_kernels.txt); None where no capture of that kernel is committed
NCU_TRAFFIC = {}
try:
    NCU_TRAFFIC = json.loads((ROOT / "profiles" / "r02_ncu_traffic.json").read_text())
except Exception:
    pass


def per_kernel_roofline(peaks, ms_per_step):
    """Live CUDA-event timings (L2 flushed before every launch) of the kernels that make up most of the step, each at
    its benchmark shape (B = 256: M = 49152 decoder rows), against the roofline SURVEY.md section 8(d) assigns: the
    tensor pipe (measured burst bf16 peak) for every dense contraction, HBM for gather / norm / loss / optimizer
    kernels.  `launches` = launches of that shape per step; share = launches * us / step time.  The entries are sorted
    by share; `roofline` in the JSON line is the first one."""
    import torch
    from m3l_b200 import ops, engine
    dev = "cuda"
    B, n, D, H, heads = BATCH_PER_GPU, 192, 256, 1024, 4
    M = B * n
    bf = lambda *shape: (torch.randn(*shape, device=dev) * 0.5).bfloat16()
    x, dy = bf(M, D), bf(M, D)
    h, dh = bf(M, H), bf(M, H)
    w1, w2 = bf(H, D) * 0.1, bf(D, H) * 0.1
    wqkv, wo = bf(3 * D, D) * 0.1, bf(D, D) * 0.1
    qkv = bf(M, 3 * D)
    gamma, beta = torch.ones(D, device=dev), torch.zeros(D, device=dev)
    b1, b2 = torch.zeros(H, device=dev), torch.zeros(D, device=dev)
    gW = torch.zeros(H, D, device=dev)
    gW2 = torch.zeros(D, H, device=dev)
    gQ = torch.zeros(3 * D, D, device=dev)
    o, lse = ops.attention_fwd(qkv, B, n, heads, 64, 0.125)
    delta = torch.zeros(M, heads, device=dev)
    st = torch.zeros(M, 2, device=dev); st[:, 1] = 1
    xo = x.clone()
    tf, hb = peaks["tf_burst"], peaks["hbm_gbs"]
    rows = []

    only = [k for k in os.environ.get("M3L_PER_KERNEL_ONLY", "").split(",") if k]     # (ncu captures of single entries)

    def add(name, fn, launches, flops=None, nbytes=None, key=None):
        if only and key not in only:
            return
        sec = time_kernel_cold(fn)
        ent = {"kernel": name, "us_per_launch": sec * 1e6, "launches_per_step": launches,
               "us_per_step": sec * 1e6 * launches, "share_of_step": sec * 1e3 * launches / ms_per_step}
        if flops is not None:
            ent.update(bound="tensor", achieved=flops / sec / 1e12, peak=tf, unit="TFLOP/s", frac=flops / sec / 1e12 / tf,
                       algorithmic_flop=flops)
        else:
            ent.update(bound="hbm", achieved=nbytes / sec / 1e9, peak=hb, unit="GB/s", frac=nbytes / sec / 1e9 / hb,
                       algorithmic_bytes=nbytes)
        ent["traffic"] = NCU_TRAFFIC.get(key or name.split()[0])
        rows.append(ent)

    # weight gradients of the decoder feed-forward (dW[1024,256] = dpre^T xn and dW[256,1024] = dx^T h): 6 per step
    add("gemm_bf16_kernel<256,1,1,4,0> wgrad dW1 = dpre^T[1024 x 49152] xn[49152 x 256]", lambda: engine.wgrad(dh, x, gW), 3,
        flops=2.0 * M * H * D, key="wgrad_ff")
    add("gemm_bf16_kernel<256,1,1,4,0> wgrad dW2 = dx^T[256 x 49152] h[49152 x 1024]", lambda: engine.wgrad(dy, h, gW2), 3,
        flops=2.0 * M * H * D, key="wgrad_ff2")
    add("gemm_bf16_kernel<256,1,1,4,0> wgrad dWqkv = dqkv^T[768 x 49152] xn[49152 x 256]", lambda: engine.wgrad(qkv, x, gQ), 3,
        flops=2.0 * M * 3 * D * D, key="wgrad_qkv")
    add("ln_mlp_fwd_kernel<1> fused LayerNorm+FF1+GELU+FF2+residual (training: stores h, GELU')",
        lambda: ops.ln_mlp_fwd(x, gamma, beta, w1, b1, w2, b2, save=True, out=xo, out_has_x=True), 3,
        flops=4.0 * M * H * D, key="ln_mlp_fwd_save")
    add("attn_bwd_kernel (B=256, n=192, 4 heads x 64)",
        lambda: ops.attention_bwd(qkv, o, dy, lse, B, n, heads, 64, 0.125, delta=delta), 3,
        flops=10.0 * n * n * 64 * B * heads, key="attn_bwd")
    add("attn_fwd_kernel (B=256, n=192, 4 heads x 64)", lambda: ops.attention_fwd(qkv, B, n, heads, 64, 0.125), 3,
        flops=4.0 * n * n * 64 * B * heads, key="attn_fwd")
    gp = h.clone()
    add("gemm_bf16_kernel<256,0,0,2,0> dgrad dpre = (dx W2) * GELU' [49152 x 1024, K=256]",
        lambda: ops.gemm(dy, w2.t().contiguous(), act=ops.GELU_BWD, aux_in=gp), 3, flops=2.0 * M * H * D, key="dgrad_ff2")
    # dgrad through FF1 / to_qkv with the LayerNorm backward (dx, dgamma, dbeta, column sums, + residual gradient) in the
    # GEMM epilogue: what used to be a dgrad GEMM + ln_bwd_pipe_kernel, six per step
    w1t, wqkvt = w1.t().contiguous(), wqkv.t().contiguous()
    dg, db, dc = (torch.zeros(D, device=dev) for _ in range(3))
    lnb = dict(x=x, stats=st, gamma=gamma, skip=dy, dgamma=dg, dbeta=db, dx_colsum=dc)
    add("gemm_bf16_kernel<256,0,0,5,0> dgrad dpre W1 + LayerNorm backward + residual gradient [49152 x 256, K=1024]",
        lambda: ops.gemm(dh, w1t, ln_bwd=lnb), 3, flops=2.0 * M * H * D, key="dgrad_ff1_ln")
    add("gemm_bf16_kernel<256,0,0,0,1> QKV projection [49152 x 768, K=256]", lambda: ops.gemm(x, wqkv), 3,
        flops=2.0 * M * 3 * D * D, key="qkv_fwd")
    add("gemm_bf16_kernel<256,0,0,0,0> attention out-projection + residual [49152 x 256, K=256]",
        lambda: ops.gemm(x, wo, bias=b2, residual=dy), 3, flops=2.0 * M * D * D, key="out_proj")
    add("ln_bwd_pipe_kernel LayerNorm backward (final decoder norm; the six per-layer ones run in GEMM epilogues) [49152 x 256]",
        lambda: ops.layernorm_bwd(dy, x, st, gamma, skip=dy), 1, nbytes=4.0 * M * D * 2 + M * 8, key="ln_bwd")
    add("ln_fwd_pipe_kernel LayerNorm forward [49152 x 256]", lambda: ops.layernorm_fwd(x, gamma, beta), 4,
        nbytes=2.0 * M * D * 2 + M * 8, key="ln_fwd")
    add("gemm_bf16_kernel<256,0,0,5,0> dgrad dqkv Wqkv + LayerNorm backward + residual gradient [49152 x 256, K=768]",
        lambda: ops.gemm(qkv, wqkvt, ln_bwd=lnb), 3, flops=2.0 * M * 3 * D * D, key="dgrad_qkv_ln")
    wot = wo.t().contiguous()
    add("gemm_bf16_kernel<256,0,0,0,0> dgrad dO = dx Wo + delta = rowsum(dO * O) per head [49152 x 256, K=256]",
        lambda: ops.gemm(dy, wot, dot_side=o, dot_out=delta), 3, flops=2.0 * M * D * D, key="out_proj_dgrad")
    rows.sort(key=lambda r: -r["share_of_step"])
    return rows


def _clocks_record(burst_sampler, sustained):
    """Clock / throttle record of the timed region.  nvidia-smi needs > 100 ms to deliver its first sample on an 8-GPU
    box, longer than the 20-step burst (~50 ms): when the burst sampler saw nothing, the record of the sustained leg
    (the same loop, >= 3 s, sampled every 100 ms) is reported and marked as such."""
    rec = burst_sampler.summary()
    if rec.get("sm_mhz") is None and sustained is not None and sustained.get("clocks", {}).get("sm_mhz") is not None:
        rec = dict(sustained["clocks"], source="sustained leg (the burst was shorter than nvidia-smi's first sample)")
    return rec


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, mae, loss):
    """What one train step hands back to its caller, as float32 DIR/<name>.npy: `loss`, and for every parameter
    `param.<name>` (the fp32 master weight after the AdamW update) and `grad.<name>` (its gradient as left in .grad,
    i.e. after clipping; only parameters the step gives a gradient).  For the benchmark model that is all of it, about
    41 MB, so nothing is sampled."""
    import numpy as np
    arrays = {"loss": loss}
    for name in mae.arena.names:
        p = mae.arena.params[name]
        arrays[f"param.{name}"] = p
        if p.grad is not None:
            arrays[f"grad.{name}"] = p.grad
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out / f"{k}.npy", a)


def _teardown(world, trainer=None):
    """Multi-rank exit: the step graphs hold captured NCCL kernels, and tearing the communicator down while they are
    alive (or letting the interpreter do it in arbitrary order at exit) can block for minutes.  Order: all ranks
    finished (barrier) -> drop the graphs -> flush -> leave the process without running the NCCL destructor path."""
    if world <= 1:
        return
    import gc
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    if trainer is not None:
        trainer._graphs.clear()
    gc.collect()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from m3l_b200.trainer import FusedTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    B = BATCH_PER_GPU
    mae = build_model(dev)
    mae._sync()
    trainer = FusedTrainer(mae, lr=1e-4, use_cuda_graph=not args.no_graph)
    mae._trainer = trainer

    # rotating resident batches: 4 x 75.5 MB inputs; together with ~2 GB of activations written per step
    # the working set is far larger than the 126 MB L2
    nbuf = 4
    host = [synth_batch(B, 1234 + rank * 100 + i, pinned=True) for i in range(nbuf)]
    devb = [({k: v.to(dev) for k, v in x.items()}, n.to(dev)) for x, n in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ------------------------------------------------------------
    for i in range(max(args.warmup, 3)):
        x, n = devb[i % nbuf]
        trainer.step(x, noise=n)
    barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        s.record()
        for i in range(args.steps):
            x, n = devb[i % nbuf]
            loss = trainer.step(x, noise=n)
        e.record()
        barrier()
    ms = s.elapsed_time(e)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = B * world * args.steps / (ms_total * 1e-3)
    loss_val = float(loss.item())
    if args.dump_outputs and rank == 0:        # replicas are identical: rank 0 speaks for all
        dump_outputs(args.dump_outputs, mae, loss)
    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms_per_step, "value": value, "loss": loss_val}), flush=True)
        _teardown(world, trainer)
        return

    # ---- sustained: the same loop for >= args.sustain_seconds (the 20-step figure above is a burst of ~50 ms)
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / ms_per_step) + 1)
        barrier()
        with ClockSampler(local) as clocks_sus:
            s.record()
            for i in range(n_sus):
                x, n = devb[i % nbuf]
                trainer.step(x, noise=n)
            e.record()
            barrier()
        t = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sustained = {"steps": n_sus, "seconds": float(t.item()) * 1e-3, "ms_per_step": float(t.item()) / n_sus,
                     "value": B * world * n_sus / (float(t.item()) * 1e-3), "clocks": clocks_sus.summary()}

    # ---- replicas: after the timed loops every rank must hold bit-identical parameters
    replicas_identical = None
    if world > 1:
        flat = mae.arena.flat
        chk = torch.stack([flat.view(torch.int32).to(torch.int64).sum(), (flat.view(torch.int32).to(torch.int64) ** 2 % 1000003).sum()])
        allc = [torch.empty_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        replicas_identical = all(torch.equal(c, allc[0]) for c in allc)

    # ---- end to end through the reference-facing call: a pinned HOST rollout batch (raw observations, as the
    #      reference's learners hold them) -> H2D every step (prefetched one step ahead on a copy stream) ->
    #      vt_load (lazy: fused into the patch-gather kernels) -> train step -> D2H read of the loss every step
    from m3l_b200.data import vt_load_lazy
    copy_stream = torch.cuda.Stream()

    def e2e_run(u8_frames):
        hostb = [synth_obs(B, 4321 + rank * 100 + i, pinned=True, u8_frames=u8_frames) for i in range(nbuf)]
        stage = [({k: torch.empty_like(v, device=dev) for k, v in hostb[0][0].items()}, torch.empty(B, 192, device=dev))
                 for _ in range(2)]
        views = [vt_load_lazy(st[0], frame_stack=4) for st in stage]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        def prefetch(i):
            slot = i % 2
            x, n = hostb[i % nbuf]
            copy_stream.wait_event(consumed[slot])
            with torch.cuda.stream(copy_stream):
                for k, v in x.items():
                    stage[slot][0][k].copy_(v, non_blocking=True)
                stage[slot][1].copy_(n, non_blocking=True)
                ready[slot].record(copy_stream)

        for ev in consumed:
            ev.record()
        h2d = sum(v.numel() * v.element_size() for v in hostb[0][0].values()) + hostb[0][1].numel() * 4
        # H2D alone (reported next to e2e: the floor the PCIe link sets for a step)
        barrier()
        hs, he = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        hs.record(copy_stream)
        for i in range(4):
            prefetch(i)
            consumed[i % 2].record(copy_stream)
        he.record(copy_stream)
        barrier()
        h2d_ms = hs.elapsed_time(he) / 4
        for ev in consumed:
            ev.record()
        for i in range(2):                                 # graph capture for this input form happens outside the timing
            prefetch(i)
            torch.cuda.current_stream().wait_event(ready[i % 2])
            trainer.step(views[i % 2], noise=stage[i % 2][1])
            consumed[i % 2].record()
        # every step's loss is copied D2H into pinned memory on the compute stream and READ by the host one
        # step later (after its event), so the host never drains the GPU queue; all K losses are read
        # inside the timed region
        k_steps = args.steps
        loss_host = torch.empty(k_steps, dtype=torch.float32).pin_memory()
        loss_ev = [torch.cuda.Event() for _ in range(k_steps)]
        barrier()
        t0 = time.perf_counter()
        s.record()
        prefetch(0)
        losses = []
        for i in range(k_steps):
            slot = i % 2
            if i + 1 < k_steps:
                prefetch(i + 1)
            torch.cuda.current_stream().wait_event(ready[slot])
            l = trainer.step(views[slot], noise=stage[slot][1])
            consumed[slot].record()
            loss_host[i:i + 1].copy_(l.reshape(1), non_blocking=True)     # D2H of the step result
            loss_ev[i].record()
            if i > 0:
                loss_ev[i - 1].synchronize()
                losses.append(float(loss_host[i - 1]))
        loss_ev[k_steps - 1].synchronize()
        losses.append(float(loss_host[k_steps - 1]))
        e.record()
        barrier()
        assert len(losses) == k_steps and all(x == x for x in losses)
        t = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return {"value": B * world * k_steps / (float(t.item()) * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "h2d_ms_per_step_alone": h2d_ms, "wall_s": time.perf_counter() - t0}

    e2e = e2e_run(False)
    e2e["note"] = ("pinned host rollout batch (raw fp32 observations: image [B,4,64,64,3], tactile [B,4,6,32,32]) -> H2D "
                   "prefetched one step ahead on a copy stream -> vt_load fused into the patch-gather kernels -> train step; "
                   "every step's loss copied D2H to pinned memory and read by the host one step later")
    e2e_u8 = e2e_run(True)
    e2e_u8["note"] = "same, with the image frames stored as uint8 in the host buffer (scaled by 1/255 inside the gather kernels)"

    if rank == 0:
        table = per_kernel_roofline(peaks, ms_per_step)
        roof = dict(table[0], peak_source=peaks["source"] + ", burst (kernel timed alone, L2 flushed)")
        step_tflops = value / world * FLOPS_PER_SAMPLE / 1e12
        # CPU baseline: rank 0 at N = 1 only (torchrun pins OMP_NUM_THREADS=1; the driver's reference arm times it)
        cpu_sps, cpu_ms, cores = cpu_reference_run(steps=30, warmup=3) if world == 1 else (None, None, None)
        launches = (trainer.kernel_launches_per_step or 0)
        line = {
            "metric": "VTMAE train samples/sec (fwd+bwd+AdamW)", "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": B * world, "batch_per_gpu": B, "parallelism": f"dp{world}",
                       "l2": "inputs rotate over 4 resident batches (302 MB) and every step streams >2 GB of "
                             "activations through HBM, far above the 126 MB L2; no explicit flush",
                       "cuda_graph": bool(trainer.use_graph), "loss_last_step": loss_val},
            "clocks": _clocks_record(clocks, sustained),
            "e2e": e2e,
            "e2e_uint8_frames": e2e_u8,
            "sustained": sustained,
            "gpu_launches": launches * args.steps,
            "gpu_launches_per_step": launches,
            "roofline": roof,
            "per_kernel": [{k: r[k] for k in ("kernel", "us_per_launch", "launches_per_step", "us_per_step", "share_of_step",
                                                "bound", "achieved", "peak", "unit", "frac", "traffic")} for r in table],
            "step_tensor_utilisation": {"achieved": step_tflops, "unit": "TFLOP/s (3404.7 MFLOP/sample x samples/s/GPU)",
                                        "peak": peaks["tf_sustained"], "frac": step_tflops / peaks["tf_sustained"],
                                        "peak_source": peaks["source"] + ", sustained"},
        }
        if replicas_identical is not None:
            line["replicas_identical"] = replicas_identical
        if cpu_sps is not None:
            line["cpu_baseline"] = {"value": cpu_sps, "unit": "samples/s", "cores": cores, "kind": "port",
                                    "sample": f"batch 32 slice of the workload, fp32 torch CPU oracle, 30 timed steps, "
                                              f"{cpu_ms:.1f} ms/step"}
        print(json.dumps(line), flush=True)
    _teardown(world, trainer)


# ------------------------------------------------------------------------------------------------
# secondary workloads of BASELINE.json (configs[2], configs[3]) - strong scaling of a fixed global batch
# ------------------------------------------------------------------------------------------------
def run_other_config(args):
    """--config 3: vision_only_control VTMAE (image tokens only), global batch 1024 split over the ranks.
    --config 4: DINO-tac-MAE variant, global batch 512: tactile-only MAE train step (70x70 maps, patch 14, dim 384)
                + the frozen DINOv2 ViT-S/14-reg forward on the mid frame of the image stack (feature branch of
                models/pretrain_models_dino_cat_mae.py:884-889; random weights: torch.hub is unreachable offline).
    value = device-resident samples/s; e2e = from pinned host rollout batches (raw observations, H2D inside)."""
    import torch
    import torch.distributed as dist
    from m3l_b200 import VTT, VTMAE
    from m3l_b200.trainer import FusedTrainer
    from m3l_b200.data import vt_load_lazy
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    torch.manual_seed(0)
    dino = None
    if args.config == 3:
        gb, flops, size, n_tok = 1024, 1140.5e6, 64, 64
        name = "vision_only_control VTMAE train step (image tokens only), global batch 1024 (BASELINE.json configs[2])"
        enc = VTT(image_size=(64, 64), tactile_size=(32, 32), image_patch_size=8, tactile_patch_size=4, dim=256, depth=4,
                  heads=4, mlp_dim=512, num_tactiles=0, image_channels=12, tactile_channels=12, frame_stack=4)
        mae = VTMAE(encoder=enc, decoder_dim=256, masking_ratio=0.95, decoder_depth=3, decoder_heads=4, num_tactiles=0,
                    frame_stack=4).to(dev)
    else:
        from m3l_b200.dinov2 import DinoV2, mid_frame_view
        gb, flops, size, n_tok = 512, 2163.5e6 + 1285.3e6, 70, 50
        name = ("DINO-tac-MAE: tactile-only VTMAE train step (70x70, patch 14, dim 384, r 0.8) + frozen DINOv2 ViT-S/14-reg "
                "forward on the mid frame, global batch 512 (BASELINE.json configs[3])")
        enc = VTT(image_size=(70, 70), tactile_size=(70, 70), image_patch_size=14, tactile_patch_size=14, dim=384, depth=4,
                  heads=4, mlp_dim=768, num_tactiles=2, image_channels=12, tactile_channels=12, frame_stack=4)
        mae = VTMAE(encoder=enc, decoder_dim=384, masking_ratio=0.8, decoder_depth=3, decoder_heads=4, num_tactiles=2,
                    frame_stack=4).to(dev)
        dino = DinoV2().to(dev).eval()
    assert gb % world == 0
    B = gb // world
    mae._sync()
    trainer = FusedTrainer(mae, lr=1e-4)

    def synth(seed):
        g = torch.Generator().manual_seed(seed)
        obs = {"image": torch.rand(B, 4, size, size, 3, generator=g).pin_memory()}
        if args.config == 4:
            obs["tactile"] = (torch.rand(B, 4, 6, size, size, generator=g) * 2 - 1).pin_memory()
        return obs, torch.rand(B, n_tok, generator=g).pin_memory()

    def step(views, noise):
        if args.config == 3:
            return trainer.step({"image": views["image"]}, noise=noise)
        loss = trainer.step({k: v for k, v in views.items() if k.startswith("tactile")}, noise=noise)
        dino(mid_frame_view(views["image"], 4))
        return loss

    nbuf = 3
    host = [synth(99 + rank * 10 + i) for i in range(nbuf)]
    devb = [(vt_load_lazy({k: v.to(dev) for k, v in o.items()}, frame_stack=4), n.to(dev)) for o, n in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:          # sampled from the warm-up on: the timed burst alone is ~50 ms
        for i in range(max(args.warmup, 3)):
            step(*devb[i % nbuf])
        barrier()
        for i in range(40):                      # ~0.15 s of the same steps so that nvidia-smi delivers samples under load
            step(*devb[i % nbuf])
        barrier()
        s.record()
        for i in range(args.steps):
            loss = step(*devb[i % nbuf])
        e.record()
        barrier()
    t = torch.tensor([s.elapsed_time(e)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = gb / (ms_per_step * 1e-3)
    # e2e: host rollout batch -> H2D (prefetched on a copy stream) -> step; loss read back every step
    copy_stream = torch.cuda.Stream()
    stage = [({k: torch.empty_like(v, device=dev) for k, v in host[0][0].items()}, torch.empty(B, n_tok, device=dev)) for _ in range(2)]
    views = [vt_load_lazy(st[0], frame_stack=4) for st in stage]
    ready, consumed = [torch.cuda.Event(), torch.cuda.Event()], [torch.cuda.Event(), torch.cuda.Event()]
    for ev in consumed:
        ev.record()

    def prefetch(i):
        slot = i % 2
        copy_stream.wait_event(consumed[slot])
        with torch.cuda.stream(copy_stream):
            for k, v in host[i % nbuf][0].items():
                stage[slot][0][k].copy_(v, non_blocking=True)
            stage[slot][1].copy_(host[i % nbuf][1], non_blocking=True)
            ready[slot].record(copy_stream)

    loss_host = torch.empty(args.steps, dtype=torch.float32).pin_memory()
    barrier()
    s.record()
    prefetch(0)
    for i in range(args.steps):
        if i + 1 < args.steps:
            prefetch(i + 1)
        torch.cuda.current_stream().wait_event(ready[i % 2])
        l = step(views[i % 2], stage[i % 2][1])
        consumed[i % 2].record()
        loss_host[i:i + 1].copy_(l.reshape(1), non_blocking=True)
    e.record()
    barrier()
    assert bool(torch.isfinite(loss_host).all())
    t = torch.tensor([s.elapsed_time(e)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = gb * args.steps / (float(t.item()) * 1e-3)
    h2d = sum(v.numel() * v.element_size() for v in host[0][0].values()) + B * n_tok * 4
    replicas_identical = None
    if world > 1:
        flat = mae.arena.flat
        chk = torch.stack([flat.view(torch.int32).to(torch.int64).sum(), (flat.view(torch.int32).to(torch.int64) ** 2 % 1000003).sum()])
        allc = [torch.empty_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        replicas_identical = all(torch.equal(c, allc[0]) for c in allc)
    if rank == 0:
        tfl = value / world * flops / 1e12
        line = {"metric": "VTMAE train samples/sec (fwd+bwd+AdamW)", "value": value, "unit": "samples/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": name, "global_batch": gb, "batch_per_gpu": B, "parallelism": f"dp{world}", "cuda_graph": True,
                           "loss_last_step": float(loss.item())},
                "clocks": clocks.summary(),
                "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
                "gpu_launches_per_step": (trainer.kernel_launches_per_step or 0) + (4 + 7 * len(dino.blocks) + 1 if dino is not None else 0),
                "step_tensor_utilisation": {"achieved": tfl, "unit": "TFLOP/s per GPU", "peak": peaks["tf_sustained"],
                                            "frac": tfl / peaks["tf_sustained"]}}
        line["gpu_launches"] = line["gpu_launches_per_step"] * args.steps
        if replicas_identical is not None:
            line["replicas_identical"] = replicas_identical
        print(json.dumps(line), flush=True)
    _teardown(world, trainer)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="m3l_b200", choices=["m3l_b200", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly (for ncu launch lists)")
    ap.add_argument("--profile", action="store_true", help="device-resident loop only (no e2e / CPU baseline legs)")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json workload: 2 = headline (configs[1]); 3 = vision-only, global batch 1024; 4 = DINO-tac-MAE, global batch 512")
    ap.add_argument("--sustain-seconds", type=float, default=3.0,
                    help="also time the device-resident loop for at least this long (0 disables)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, parameters and gradients of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "m3l_b200" or args.config != 2):
        ap.error("--dump-outputs is available for the headline workload (--config 2, --impl m3l_b200)")
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.config in (3, 4):
        run_other_config(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
