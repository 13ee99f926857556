"""DinoV2 fine-tuning: forward + backward of m3l_b200.DinoV2 (training mode, CUDA graphs) against `transformers`
Dinov2WithRegistersModel in bf16 autocast with SDPA attention, on the same GPU, same weights shape (dinov2_vits14_reg,
518 x 518 position table, so both inputs below go through the position interpolation).

Shapes: B = 64 at 224 x 224 (n = 261 tokens) and B = 512 at 70 x 70 (n = 30), all blocks trainable and the last 4
blocks trainable (the rest of the network frozen, requires_grad False).  A step is forward, a random cotangent on the
class token, backward and zero_grad(set_to_none=True); the time per step is the median of 5 CUDA-event windows of
20 steps after 10 warm-up steps.  The card's name and power limit are read in the same call.

    python tools/bench_dinov2_train.py --out /tmp/r06_bench_dinov2_train.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_long_attention import gpu_info  # noqa: E402

SHAPES = [(64, 224), (512, 70)]
LAST = 4


def time_steps(step, warmup=10, steps=20, windows=5):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    ms = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b) / steps)
    return statistics.median(ms), ms


def set_trainable(named, depth, prefix, last):
    for k, p in named:
        if last is None:
            p.requires_grad_(True)
        else:
            parts = k.split(".")
            p.requires_grad_(k.startswith(prefix) and int(parts[len(prefix.split(".")) - 1]) >= depth - last)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_bench_dinov2_train.json"))
    ap.add_argument("--shapes", default=",".join(f"{b}x{s}" for b, s in SHAPES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dinov2_train.py needs a CUDA device")
    import transformers as tr
    from m3l_b200.dinov2 import DinoV2
    from oracle import dinov2_oracle as DO

    torch.manual_seed(0)
    sd = DO.random_state_dict(grid=37, seed=0)
    sd["mask_token"] = torch.zeros(1, 384)
    ours = DinoV2()
    ours.load_state_dict(sd)
    ours = ours.cuda().train()
    cfg = tr.Dinov2WithRegistersConfig(hidden_size=384, num_hidden_layers=12, num_attention_heads=6, mlp_ratio=4,
                                       patch_size=14, image_size=518, num_register_tokens=4, layerscale_value=1.0,
                                       attn_implementation="sdpa")
    ref = tr.Dinov2WithRegistersModel(cfg).cuda().train()
    depth = 12
    rows = []
    for shape in args.shapes.split(","):
        B, S = (int(v) for v in shape.split("x"))
        x = torch.rand(B, 3, S, S, device="cuda")
        cot = torch.randn(B, 384, device="cuda")
        n = 1 + 4 + (S // 14) ** 2
        for last in (None, LAST):
            set_trainable(ours.named_parameters(), depth, "blocks.", last)
            set_trainable(ref.named_parameters(), depth, "encoder.layer.", last)

            def step_ours():
                (ours(x) * cot).sum().backward()
                ours.zero_grad(set_to_none=True)

            def step_ref():
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    out = ref(pixel_values=x).pooler_output
                (out.float() * cot).sum().backward()
                ref.zero_grad(set_to_none=True)

            t_ours, w_ours = time_steps(step_ours)
            t_ref, w_ref = time_steps(step_ref)
            row = {"batch": B, "image": S, "tokens": n, "trainable": "all blocks" if last is None else f"last {last} blocks",
                   "m3l_ms_per_step": t_ours, "transformers_bf16_sdpa_ms_per_step": t_ref,
                   "speedup": t_ref / t_ours, "m3l_samples_per_s": B / t_ours * 1e3,
                   "transformers_samples_per_s": B / t_ref * 1e3, "m3l_windows_ms": w_ours, "transformers_windows_ms": w_ref}
            print(json.dumps(row), flush=True)
            rows.append(row)
    res = {"what": "DinoV2 fine-tuning forward + backward per step (tools/bench_dinov2_train.py)", "gpu": gpu_info(),
           "torch": torch.__version__, "transformers": tr.__version__, "rows": rows}
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
