"""Attention kernels and the VTMAE train step at head widths 32, 64 and 128 for equal `inner` = heads * dim_head.

Kernel part: for each shape, the forward and backward of the kernel family that ops.mha_fwd / mha_bwd pick for that
width (64: attention.cu up to 256 tokens, attention_long.cu above; 32 / 128: attention_dh.cu at every length) against
torch's scaled_dot_product_attention on the same bf16 tensors.  Every kernel time is the median of 20 CUDA-event
timings of single launches, each preceded by a 256 MB write that evicts the 126 MB L2; every shape is warmed up
before its timed passes.  FLOPs per (sample, head) as in DESIGN.md: 4 n^2 dh forward, 10 n^2 dh backward.  The
backward runs with delta = rowsum(dO * O) supplied where the model code supplies it (dh = 64) and computes it in the
kernel otherwise, as the model code does.

Train-step part: FusedTrainer samples/s at the bench.py shape (batch 256, 64 x 64 image + two 32 x 32 tactile maps,
encoder depth 4, decoder depth 3, dim 256) with encoder and decoder both at (heads 8, dh 32), (4, 64) and (2, 128).
CUDA graph on, median of 5 windows of 20 steps after 10 warm-up steps.

Prints one JSON object (and writes it to --out).

    python tools/bench_head_dims.py --out /tmp/bench_head_dims.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_long_attention import PEAK_TFLOPS, Timer, gpu_info, sdpa_backend  # noqa: E402

INNER = 256
SHAPES = [  # (B, n, where from)
    (256, 10, "VTMAE masked encoder (cfg 2)"),
    (256, 192, "VTMAE decoder (cfg 2)"),
    (256, 384, "VTMAE 128 x 128 image decoder"),
    (64, 1374, "DinoV2 @518 length"),
]
WIDTHS = (32, 64, 128)


def bench_shape(ops, timer, B, n, dh, where):
    torch.manual_seed(0)
    H = INNER // dh
    scale = dh ** -0.5
    qkv = torch.randn(B * n, 3 * INNER, device="cuda").bfloat16()
    dout = torch.randn(B * n, INNER, device="cuda").bfloat16()
    fl_fwd, fl_bwd = 4 * n * n * dh * B * H, 10 * n * n * dh * B * H
    row = {"B": B, "n": n, "H": H, "dim_head": dh, "from": where}

    def rate(us, flops):
        tf = flops / (us * 1e-6) / 1e12
        return {"us": round(us, 2), "tflops": round(tf, 2), "share_of_peak": round(tf / PEAK_TFLOPS, 4)}

    out = torch.empty(B * n, INNER, dtype=torch.bfloat16, device="cuda")
    lse = torch.empty(B, H, n, dtype=torch.float32, device="cuda")
    ops.mha_fwd(qkv, B, n, H, dh, scale, out=out, lse=lse)
    delta = (dout.float() * out.float()).reshape(B * n, H, dh).sum(-1).contiguous() if dh == 64 else None
    dqkv = torch.empty_like(qkv)
    fam = "attention_dh" if dh != 64 else ("attention" if n <= ops.SHORT_ATTENTION_MAX_N else "attention_long")
    t_f = timer(lambda: ops.mha_fwd(qkv, B, n, H, dh, scale, out=out, lse=lse))
    t_b = timer(lambda: ops.mha_bwd(qkv, out, dout, lse, B, n, H, dh, scale, dqkv=dqkv, delta=delta))
    row["m3l"] = {"kernels": fam, "bwd_delta": "supplied" if delta is not None else "in kernel",
                  "fwd": rate(t_f, fl_fwd), "bwd": rate(t_b, fl_bwd)}
    qkv5 = qkv.view(B, n, 3, H, dh).detach().requires_grad_(True)
    q, k, v = (t.transpose(1, 2) for t in qkv5.unbind(2))
    o = F.scaled_dot_product_attention(q, k, v, scale=scale)
    do = dout.view(B, n, H, dh).transpose(1, 2)
    fwd = lambda: F.scaled_dot_product_attention(q, k, v, scale=scale)      # noqa: E731
    bwd = lambda: torch.autograd.grad(o, qkv5, do, retain_graph=True)       # noqa: E731
    backend_f, _ = sdpa_backend(fwd)
    backend_b, _ = sdpa_backend(bwd)
    row["sdpa"] = {"fwd": rate(timer(fwd), fl_fwd), "bwd": rate(timer(bwd), fl_bwd), "backend_fwd": backend_f,
                   "backend_bwd": backend_b}
    return row


def bench_train(heads, dh, B=256, warm=10, steps=20, windows=5):
    from m3l_b200 import VTT, VTMAE
    from m3l_b200.trainer import FusedTrainer
    torch.manual_seed(0)
    enc = VTT(image_size=(64, 64), tactile_size=(32, 32), image_patch_size=8, tactile_patch_size=4, dim=256, depth=4,
              heads=heads, dim_head=dh, mlp_dim=512, num_tactiles=2, image_channels=12, tactile_channels=12,
              frame_stack=4)
    mae = VTMAE(encoder=enc, decoder_dim=256, masking_ratio=0.95, decoder_depth=3, decoder_heads=heads,
                decoder_dim_head=dh, num_tactiles=2, early_conv_masking=False, frame_stack=4).cuda()
    mae._sync()
    trainer = FusedTrainer(mae, lr=1e-4)
    mae._trainer = trainer
    g = torch.Generator().manual_seed(1234)
    bufs = []
    for _ in range(4):
        x = {"image": torch.rand(B, 12, 64, 64, generator=g), "tactile1": torch.rand(B, 12, 32, 32, generator=g),
             "tactile2": torch.rand(B, 12, 32, 32, generator=g)}
        bufs.append(({k: v.cuda() for k, v in x.items()}, torch.rand(B, 192, generator=g).cuda()))
    for i in range(warm):
        x, n = bufs[i % 4]
        trainer.step(x, noise=n)
    torch.cuda.synchronize()
    rates = []
    for _ in range(windows):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            x, n = bufs[i % 4]
            loss = trainer.step(x, noise=n)
        e.record()
        e.synchronize()
        rates.append(B * steps / (s.elapsed_time(e) * 1e-3))
    res = {"encoder": [heads, dh], "decoder": [heads, dh], "samples_per_s": round(statistics.median(rates), 1),
           "windows": [round(r, 1) for r in rates], "loss": float(loss.item())}
    del trainer, mae
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    from m3l_b200 import ops
    timer = Timer()
    res = {"gpu": gpu_info(), "torch": torch.__version__, "peak_tflops_bf16_measured": PEAK_TFLOPS, "inner": INNER,
           "l2": "256 MB buffer written before every timed launch", "reps": 20,
           "kernels": [bench_shape(ops, timer, B, n, dh, where) for B, n, where in SHAPES for dh in WIDTHS],
           "train_step_cfg2": [bench_train(INNER // dh, dh) for dh in WIDTHS]}
    res["gpu_after"] = gpu_info()
    text = json.dumps(res)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
