"""Attention kernels at sequence lengths around and above 256 tokens, against torch's scaled_dot_product_attention,
and DinoV2 end to end at 224 x 224 against `transformers`' Dinov2WithRegistersModel (bf16, SDPA).

Every kernel time is the median of CUDA-event timings of single launches, each preceded by a 256 MB write that
evicts the 126 MB L2; every shape is warmed up before its timed passes.  FLOPs per (sample, head) are counted as
in DESIGN.md: 4 n^2 64 forward, 10 n^2 64 backward (recomputed S included).  The share of peak is against the
measured dense bf16 rate of DESIGN.md (1684.2 TFLOP/s).  The backward runs with delta = rowsum(dO * O) supplied,
as the model code calls it.  Prints one JSON object (and writes it to --out).

    python tools/bench_long_attention.py --out /tmp/bench_long_attention.json
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

PEAK_TFLOPS = 1684.2
SHAPES = [  # (B, n, H, where from)
    (256, 261, 6, "DinoV2 @224"),
    (64, 1374, 6, "DinoV2 @518"),
    (256, 384, 4, "VTMAE 128x128 image decoder"),
    (32, 1024, 4, "longer sequence"),
    (8, 4096, 4, "longer sequence"),
    (256, 192, 4, "both kernels (n <= 256)"),
    (256, 256, 4, "both kernels (n <= 256)"),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = [s.strip() for s in q[0].split(",")] if q else (torch.cuda.get_device_name(), "?", "?")
    return {"name": name, "power_limit": power, "sm_max_clock": clk}


class Timer:
    def __init__(self):
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def __call__(self, fn, reps=20, warmup=3):
        for _ in range(warmup):
            fn()
        times = []
        for _ in range(reps):
            self.flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) * 1e3)
        times.sort()
        return times[len(times) // 2]


def sdpa_backend(fn):
    """Names of the CUDA kernels one call launches, and the SDPA backend they belong to."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA})
    joined = " ".join(names).lower()
    if "cudnn" in joined or "sm100_" in joined or "cudnn_generated" in joined:
        backend = "cudnn"
    elif "flash" in joined:
        backend = "flash"
    elif "fmha" in joined or "efficient" in joined or "cutlass" in joined:
        backend = "efficient"
    else:
        backend = "math"
    return backend, names


def bench_shape(ops, timer, B, n, H, where):
    torch.manual_seed(0)
    scale = 64 ** -0.5
    inner = H * 64
    qkv = torch.randn(B * n, 3 * inner, device="cuda").bfloat16()
    dout = torch.randn(B * n, inner, device="cuda").bfloat16()
    fl_fwd, fl_bwd = 4 * n * n * 64 * B * H, 10 * n * n * 64 * B * H
    row = {"B": B, "n": n, "H": H, "from": where}

    def rate(us, flops):
        tf = flops / (us * 1e-6) / 1e12
        return {"us": round(us, 2), "tflops": round(tf, 1), "share_of_peak": round(tf / PEAK_TFLOPS, 3)}

    kernels = [("long", ops.attention_long_fwd, ops.attention_long_bwd)]
    if n <= ops.SHORT_ATTENTION_MAX_N:
        kernels.append(("short", ops.attention_fwd, ops.attention_bwd))
    for name, f, bw in kernels:
        out = torch.empty(B * n, inner, dtype=torch.bfloat16, device="cuda")
        lse = torch.empty(B, H, n, dtype=torch.float32, device="cuda")
        f(qkv, B, n, H, 64, scale, out=out, lse=lse)
        delta = (dout.float() * out.float()).reshape(B * n, H, 64).sum(-1).contiguous()
        dqkv = torch.empty_like(qkv)
        t_f = timer(lambda: f(qkv, B, n, H, 64, scale, out=out, lse=lse))
        t_b = timer(lambda: bw(qkv, out, dout, lse, B, n, H, 64, scale, dqkv=dqkv, delta=delta))
        row[name] = {"fwd": rate(t_f, fl_fwd), "bwd": rate(t_b, fl_bwd)}
    # torch SDPA on the same bf16 tensors ([B, H, n, 64] views of the packed qkv)
    qkv5 = qkv.view(B, n, 3, H, 64).detach().requires_grad_(True)
    q, k, v = (t.transpose(1, 2) for t in qkv5.unbind(2))
    o = F.scaled_dot_product_attention(q, k, v, scale=scale)
    do = dout.view(B, n, H, 64).transpose(1, 2)
    fwd = lambda: F.scaled_dot_product_attention(q, k, v, scale=scale)      # noqa: E731
    bwd = lambda: torch.autograd.grad(o, qkv5, do, retain_graph=True)       # noqa: E731
    backend_f, names_f = sdpa_backend(fwd)
    backend_b, names_b = sdpa_backend(bwd)
    row["sdpa"] = {"fwd": rate(timer(fwd), fl_fwd), "bwd": rate(timer(bwd), fl_bwd), "backend_fwd": backend_f,
                   "backend_bwd": backend_b, "kernels_fwd": names_f, "kernels_bwd": names_b}
    return row


def bench_dinov2(timer, B=256, size=224):
    from m3l_b200.dinov2 import DinoV2
    from oracle import dinov2_oracle as DO
    torch.manual_seed(0)
    x = torch.rand(B, 3, size, size, device="cuda")
    sd = DO.random_state_dict(grid=37, seed=0)
    sd["mask_token"] = torch.zeros(1, 384)
    ours = DinoV2()
    ours.load_state_dict(sd)
    ours = ours.cuda().eval()
    with torch.no_grad():
        t_ours = timer(lambda: ours(x), reps=10)
    res = {"B": B, "size": size, "tokens": 1 + 4 + (size // 14) ** 2,
           "m3l_b200": {"ms": round(t_ours / 1e3, 3), "images_per_s": round(B / (t_ours * 1e-6), 1)}}
    del ours
    try:
        import transformers as tr
    except ImportError:
        res["transformers"] = "not installed"
        return res
    cfg = tr.Dinov2WithRegistersConfig(hidden_size=384, num_hidden_layers=12, num_attention_heads=6, mlp_ratio=4,
                                       patch_size=14, image_size=518, num_register_tokens=4, attn_implementation="sdpa")
    ref = tr.Dinov2WithRegistersModel(cfg).to(device="cuda", dtype=torch.bfloat16).eval()
    xb = x.bfloat16()
    with torch.no_grad():
        t_ref = timer(lambda: ref(pixel_values=xb), reps=10)
    res["transformers"] = {"ms": round(t_ref / 1e3, 3), "images_per_s": round(B / (t_ref * 1e-6), 1),
                           "model": "Dinov2WithRegistersModel, random weights, bf16, attn_implementation=sdpa",
                           "transformers_version": tr.__version__}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    from m3l_b200 import ops
    timer = Timer()
    res = {"gpu": gpu_info(), "torch": torch.__version__, "peak_tflops_bf16_measured": PEAK_TFLOPS,
           "l2": "256 MB buffer written before every timed launch", "bwd_delta": "supplied",
           "shapes": [bench_shape(ops, timer, *s) for s in SHAPES], "dinov2_e2e": bench_dinov2(timer)}
    res["gpu_after"] = gpu_info()
    text = json.dumps(res)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
