"""Cost of dropout in training mode: the dropout kernels at p = 0.1 against what runs at p = 0.

Kernel part: attention forward and backward through ops.mha_fwd / mha_bwd, without dropout (attention.cu up to 256
tokens at dh = 64, attention_long.cu above, attention_dh.cu for 32 / 128) and with dropout (attention_dropout.cu at
every length), for dh = 64 and for dh = 32 / 128 at the same inner width (256); and the two dropout GEMM epilogues
(GELU, bias + residual) against the plain ones at the cfg 2 encoder shapes.  Every kernel time is the median of 20
CUDA-event timings of single launches, each preceded by a 256 MB write that evicts the 126 MB L2.

Train-step part: FusedTrainer samples/s at the bench.py cfg 2 shape with encoder dropout 0.1 and 0 (CUDA graph on,
median of 5 windows of 20 steps after 10 warm-up steps).

    python tools/bench_dropout.py --out /tmp/bench_dropout.json
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

from bench_long_attention import Timer, gpu_info  # noqa: E402

INNER = 256
P = 0.1
SHAPES = [(256, 10, "VTMAE masked encoder (cfg 2)"), (256, 192, "VTMAE decoder (cfg 2)"),
          (256, 384, "VTMAE 128 x 128 image decoder"), (64, 1374, "DinoV2 @518 length")]


def bench_attention(ops, timer, B, n, dh, where):
    torch.manual_seed(0)
    H = INNER // dh
    scale = dh ** -0.5
    qkv = torch.randn(B * n, 3 * INNER, device="cuda").bfloat16()
    dout = torch.randn(B * n, INNER, device="cuda").bfloat16()
    out = torch.empty(B * n, INNER, dtype=torch.bfloat16, device="cuda")
    lse = torch.empty(B, H, n, dtype=torch.float32, device="cuda")
    dqkv = torch.empty_like(qkv)
    key = torch.tensor([12345], dtype=torch.int64, device="cuda")
    ops.mha_fwd(qkv, B, n, H, dh, scale, out=out, lse=lse)
    delta = (dout.float() * out.float()).reshape(B * n, H, dh).sum(-1).contiguous() if dh == 64 else None
    row = {"B": B, "n": n, "H": H, "dim_head": dh, "from": where}
    for name, d in (("p0", None), ("p0.1", ops.Dropout(key, 0, P))):
        f = timer(lambda: ops.mha_fwd(qkv, B, n, H, dh, scale, out=out, lse=lse, dropout=d))
        b = timer(lambda: ops.mha_bwd(qkv, out, dout, lse, B, n, H, dh, scale, dqkv=dqkv, delta=delta, dropout=d))
        row[name] = {"fwd_us": round(f, 2), "bwd_us": round(b, 2)}
    row["ratio_fwd"] = round(row["p0.1"]["fwd_us"] / row["p0"]["fwd_us"], 3)
    row["ratio_bwd"] = round(row["p0.1"]["bwd_us"] / row["p0"]["bwd_us"], 3)
    return row


def bench_gemm(ops, timer, M=2560):
    """Encoder feed-forward of cfg 2 (256 samples x 10 visible tokens, dim 256, mlp 512) and its attention output."""
    torch.manual_seed(0)
    key = torch.tensor([777], dtype=torch.int64, device="cuda")
    rows = []
    for name, K, N in (("ff1_gelu", 256, 512), ("ff2_residual", 512, 256), ("to_out_residual", 256, 256)):
        a = torch.randn(M, K, device="cuda").bfloat16()
        w = (torch.randn(N, K, device="cuda") * 0.05).bfloat16()
        bias = torch.randn(N, device="cuda") * 0.1
        res = torch.randn(M, N, device="cuda").bfloat16()
        aux = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
        out = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
        kw = dict(act=ops.GELU_FWD, aux_out=aux) if name == "ff1_gelu" else dict(residual=res)
        t0 = timer(lambda: ops.gemm(a, w, bias=bias, out=out, **kw))
        t1 = timer(lambda: ops.gemm(a, w, bias=bias, out=out, dropout=ops.Dropout(key, 2, P), **kw))
        rows.append({"gemm": name, "M": M, "K": K, "N": N, "p0_us": round(t0, 2), "p0.1_us": round(t1, 2),
                     "ratio": round(t1 / t0, 3)})
    return rows


def bench_train(p, B=256, warm=10, steps=20, windows=5):
    from m3l_b200 import VTT, VTMAE
    from m3l_b200.trainer import FusedTrainer
    torch.manual_seed(0)
    enc = VTT(image_size=(64, 64), tactile_size=(32, 32), image_patch_size=8, tactile_patch_size=4, dim=256, depth=4,
              heads=4, dim_head=64, mlp_dim=512, num_tactiles=2, image_channels=12, tactile_channels=12,
              frame_stack=4, dropout=p)
    mae = VTMAE(encoder=enc, decoder_dim=256, masking_ratio=0.95, decoder_depth=3, decoder_heads=4,
                decoder_dim_head=64, num_tactiles=2, early_conv_masking=False, frame_stack=4).cuda()
    mae.train()
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
    res = {"encoder_dropout": p, "samples_per_s": round(statistics.median(rates), 1),
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
    res = {"gpu": gpu_info(), "torch": torch.__version__, "p": P, "inner": INNER,
           "l2": "256 MB buffer written before every timed launch", "reps": 20,
           "attention": [bench_attention(ops, timer, B, n, dh, where) for B, n, where in SHAPES for dh in (32, 64, 128)],
           "gemm": bench_gemm(ops, timer),
           "train_step_cfg2": [bench_train(p) for p in (0.0, P, 0.0, P)]}
    res["gpu_after"] = gpu_info()
    text = json.dumps(res)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
