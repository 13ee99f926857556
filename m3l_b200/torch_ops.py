"""`torch.library` registration of the C-ABI entry points: namespace `m3l`.

This is the "thin C-ABI PyTorch custom-op layer" of the boundary (SURVEY.md §8b): every op below is a functional
wrapper (fresh outputs, no aliasing) around one C-ABI kernel of include/m3l_b200.h, registered with
  * a schema (`torch.ops.m3l.<name>`),
  * a CUDA implementation that hands raw device pointers + the current stream to libm3l_b200.so (ctypes loader),
  * a fake / meta implementation (shapes and dtypes only) so the ops trace under FakeTensorMode / torch.export /
    `torch.library.opcheck`,
and no CPU implementation: calling one with CPU tensors raises NotImplementedError from the dispatcher — there is no
CPU fallback anywhere in the product.

What each op stands in for in the reference (paths under /root/reference):
  m3l::linear         nn.Linear forward / dgrad with fused bias, residual, GELU / ReLU  (vit_pytorch Attention /
                      FeedForward via models/pretrain_models.py:113,784; patch embedding :769-778; heads :115-116)
  m3l::wgrad          nn.Linear weight gradient dW = dY^T X
  m3l::layernorm_fwd / layernorm_bwd      nn.LayerNorm (vit_pytorch blocks, patch embedding, final norms)
  m3l::attention_fwd / attention_bwd      softmax(q k^T / sqrt(d)) v of vit_pytorch.Attention, fused (n <= 256)
  m3l::attention_long_fwd / attention_long_bwd   the same for any sequence length (online softmax over key tiles)
  m3l::attention_dh_fwd / attention_dh_bwd       the same for 32- and 128-wide heads, any sequence length
  m3l::attention_dropout_fwd / attention_dropout_bwd   the same with Attention.dropout on the probabilities (training)
  m3l::dropout_bwd    backward of a Dropout applied in a GEMM epilogue (FeedForward / Attention.to_out Dropout)
  m3l::ln_mlp_fwd / ln_mlp_bwd            x + FeedForward(x) of vit_pytorch.Transformer as one kernel each way
  m3l::mask_indices   torch.rand(...).argsort() split into masked / unmasked (models/pretrain_models.py:229-248)
  m3l::patch_layernorm                    Rearrange('b c (h p1) (w p2) -> b (h w) (p1 p2 c)') + gather + LayerNorm (:164-198,766-779)
  m3l::masked_patch_mse                   F.mse_loss(pred, patches[batch, masked]) and its gradient (:261-262,336-340)
  m3l::vt_load        utils/pretrain_utils.py:7-57 (+ the 5-D frame-stack reshape, models/pretrain_models.py:823-827)

The module-level composition (m3l_b200.engine) calls the same kernels through m3l_b200.ops with preallocated
outputs and in-place accumulation, which a functional op schema cannot express; both layers bind the same symbols.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import ops

_lib = torch.library.Library("m3l", "DEF")
_NAMES: List[str] = []


def _define(schema: str, cuda_impl, fake_impl):
    name = schema.split("(")[0]
    _lib.define(schema)
    _lib.impl(name, cuda_impl, "CUDA")
    torch.library.register_fake(f"m3l::{name}", fake_impl, lib=_lib)
    _NAMES.append(name)


def registered_ops() -> Tuple[str, ...]:
    return tuple(_NAMES)


# ---------------------------------------------------------------------------------------------- linear / wgrad
def _linear(a: Tensor, w: Tensor, bias: Optional[Tensor] = None, residual: Optional[Tensor] = None, act: int = 0,
            out_fp32: bool = False) -> Tensor:
    return ops.gemm(a.contiguous(), w.contiguous(), bias=bias, residual=residual, act=act,
                    out_dtype=torch.float32 if out_fp32 else torch.bfloat16)


def _linear_fake(a, w, bias=None, residual=None, act=0, out_fp32=False):
    torch._check(a.dim() == 2 and w.dim() == 2 and a.shape[1] == w.shape[1], lambda: "linear: a [M, K], w [N, K]")
    torch._check(a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16, lambda: "linear: bf16 operands")
    return a.new_empty((a.shape[0], w.shape[0]), dtype=torch.float32 if out_fp32 else torch.bfloat16)


_define("linear(Tensor a, Tensor w, Tensor? bias=None, Tensor? residual=None, int act=0, bool out_fp32=False) -> Tensor",
        _linear, _linear_fake)


def _wgrad(dy: Tensor, x: Tensor) -> Tensor:
    from .engine import _wgrad_tiling
    bn, splits = _wgrad_tiling(dy.shape[1], x.shape[1], dy.shape[0])
    return ops.gemm(dy.contiguous(), x.contiguous(), mn_major=True, accumulate=True, splits=splits, bn=bn)


def _wgrad_fake(dy, x):
    torch._check(dy.dim() == 2 and x.dim() == 2 and dy.shape[0] == x.shape[0], lambda: "wgrad: dy [M, out], x [M, in]")
    return dy.new_empty((dy.shape[1], x.shape[1]), dtype=torch.float32)


_define("wgrad(Tensor dy, Tensor x) -> Tensor", _wgrad, _wgrad_fake)


# ---------------------------------------------------------------------------------------------- LayerNorm
def _ln_fwd(x: Tensor, gamma: Tensor, beta: Tensor, eps: float = 1e-5) -> Tuple[Tensor, Tensor]:
    out, stats = ops.layernorm_fwd(x.contiguous(), gamma, beta, eps=eps, want_stats=True)
    return out, stats


def _ln_fwd_fake(x, gamma, beta, eps=1e-5):
    torch._check(x.dim() == 2 and gamma.shape == (x.shape[1],) and beta.shape == (x.shape[1],), lambda: "layernorm_fwd: x [M, D]")
    return x.new_empty(x.shape, dtype=torch.bfloat16), x.new_empty((x.shape[0], 2), dtype=torch.float32)


_define("layernorm_fwd(Tensor x, Tensor gamma, Tensor beta, float eps=1e-5) -> (Tensor, Tensor)", _ln_fwd, _ln_fwd_fake)


def _ln_bwd(dy: Tensor, x: Tensor, stats: Tensor, gamma: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    D = x.shape[1]
    dgamma = torch.zeros(D, dtype=torch.float32, device=x.device)
    dbeta = torch.zeros(D, dtype=torch.float32, device=x.device)
    dx = ops.layernorm_bwd(dy.contiguous(), x.contiguous(), stats, gamma, dgamma=dgamma, dbeta=dbeta)
    return dx, dgamma, dbeta


def _ln_bwd_fake(dy, x, stats, gamma):
    torch._check(dy.shape == x.shape and stats.shape == (x.shape[0], 2), lambda: "layernorm_bwd: shapes")
    D = x.shape[1]
    return (x.new_empty(x.shape, dtype=torch.bfloat16), x.new_empty((D,), dtype=torch.float32),
            x.new_empty((D,), dtype=torch.float32))


_define("layernorm_bwd(Tensor dy, Tensor x, Tensor stats, Tensor gamma) -> (Tensor, Tensor, Tensor)", _ln_bwd, _ln_bwd_fake)


# ---------------------------------------------------------------------------------------------- attention
def _attn_fwd(qkv: Tensor, batch: int, n: int, heads: int, dim_head: int, scale: float) -> Tuple[Tensor, Tensor]:
    return ops.attention_fwd(qkv.contiguous(), batch, n, heads, dim_head, scale)


def _attn_fwd_fake(qkv, batch, n, heads, dim_head, scale):
    inner = heads * dim_head
    torch._check(qkv.shape == (batch * n, 3 * inner) and qkv.dtype == torch.bfloat16, lambda: "attention_fwd: qkv [B*n, 3*h*d] bf16")
    return qkv.new_empty((batch * n, inner)), qkv.new_empty((batch, heads, n), dtype=torch.float32)


_define("attention_fwd(Tensor qkv, int batch, int n, int heads, int dim_head, float scale) -> (Tensor, Tensor)",
        _attn_fwd, _attn_fwd_fake)


def _attn_bwd(qkv: Tensor, out: Tensor, dout: Tensor, lse: Tensor, batch: int, n: int, heads: int, dim_head: int,
              scale: float) -> Tensor:
    return ops.attention_bwd(qkv.contiguous(), out.contiguous(), dout.contiguous(), lse, batch, n, heads, dim_head, scale)


def _attn_bwd_fake(qkv, out, dout, lse, batch, n, heads, dim_head, scale):
    torch._check(out.shape == dout.shape and qkv.shape[0] == out.shape[0], lambda: "attention_bwd: shapes")
    return qkv.new_empty(qkv.shape)


_define("attention_bwd(Tensor qkv, Tensor out, Tensor dout, Tensor lse, int batch, int n, int heads, int dim_head, "
        "float scale) -> Tensor", _attn_bwd, _attn_bwd_fake)


def _attn_long_fwd(qkv: Tensor, batch: int, n: int, heads: int, dim_head: int, scale: float) -> Tuple[Tensor, Tensor]:
    return ops.attention_long_fwd(qkv.contiguous(), batch, n, heads, dim_head, scale)


_define("attention_long_fwd(Tensor qkv, int batch, int n, int heads, int dim_head, float scale) -> (Tensor, Tensor)",
        _attn_long_fwd, _attn_fwd_fake)


def _attn_long_bwd(qkv: Tensor, out: Tensor, dout: Tensor, lse: Tensor, batch: int, n: int, heads: int, dim_head: int,
                   scale: float) -> Tensor:
    return ops.attention_long_bwd(qkv.contiguous(), out.contiguous(), dout.contiguous(), lse.contiguous(), batch, n, heads,
                                  dim_head, scale)


_define("attention_long_bwd(Tensor qkv, Tensor out, Tensor dout, Tensor lse, int batch, int n, int heads, int dim_head, "
        "float scale) -> Tensor", _attn_long_bwd, _attn_bwd_fake)


def _attn_dh_fwd(qkv: Tensor, batch: int, n: int, heads: int, dim_head: int, scale: float) -> Tuple[Tensor, Tensor]:
    return ops.attention_dh_fwd(qkv.contiguous(), batch, n, heads, dim_head, scale)


_define("attention_dh_fwd(Tensor qkv, int batch, int n, int heads, int dim_head, float scale) -> (Tensor, Tensor)",
        _attn_dh_fwd, _attn_fwd_fake)


def _attn_dh_bwd(qkv: Tensor, out: Tensor, dout: Tensor, lse: Tensor, batch: int, n: int, heads: int, dim_head: int,
                 scale: float) -> Tensor:
    return ops.attention_dh_bwd(qkv.contiguous(), out.contiguous(), dout.contiguous(), lse.contiguous(), batch, n, heads,
                                dim_head, scale)


_define("attention_dh_bwd(Tensor qkv, Tensor out, Tensor dout, Tensor lse, int batch, int n, int heads, int dim_head, "
        "float scale) -> Tensor", _attn_dh_bwd, _attn_bwd_fake)


def _attn_dropout_fwd(qkv: Tensor, batch: int, n: int, heads: int, dim_head: int, scale: float, key: Tensor, site: int,
                      p: float) -> Tuple[Tensor, Tensor]:
    return ops.attention_dropout_fwd(qkv.contiguous(), batch, n, heads, dim_head, scale, ops.Dropout(key, site, p))


def _attn_dropout_fwd_fake(qkv, batch, n, heads, dim_head, scale, key, site, p):
    return _attn_fwd_fake(qkv, batch, n, heads, dim_head, scale)


_define("attention_dropout_fwd(Tensor qkv, int batch, int n, int heads, int dim_head, float scale, Tensor key, int site, "
        "float p) -> (Tensor, Tensor)", _attn_dropout_fwd, _attn_dropout_fwd_fake)


def _attn_dropout_bwd(qkv: Tensor, out: Tensor, dout: Tensor, lse: Tensor, batch: int, n: int, heads: int, dim_head: int,
                      scale: float, key: Tensor, site: int, p: float) -> Tensor:
    return ops.attention_dropout_bwd(qkv.contiguous(), out.contiguous(), dout.contiguous(), lse.contiguous(), batch, n,
                                     heads, dim_head, scale, ops.Dropout(key, site, p))


def _attn_dropout_bwd_fake(qkv, out, dout, lse, batch, n, heads, dim_head, scale, key, site, p):
    return _attn_bwd_fake(qkv, out, dout, lse, batch, n, heads, dim_head, scale)


_define("attention_dropout_bwd(Tensor qkv, Tensor out, Tensor dout, Tensor lse, int batch, int n, int heads, "
        "int dim_head, float scale, Tensor key, int site, float p) -> Tensor", _attn_dropout_bwd, _attn_dropout_bwd_fake)


def _dropout_bwd(dy: Tensor, key: Tensor, site: int, p: float) -> Tensor:
    return ops.dropout_bwd(dy.contiguous(), ops.Dropout(key, site, p))


def _dropout_bwd_fake(dy, key, site, p):
    torch._check(dy.dim() == 2 and dy.dtype == torch.bfloat16, lambda: "dropout_bwd: dy [rows, cols] bf16")
    return dy.new_empty(dy.shape)


_define("dropout_bwd(Tensor dy, Tensor key, int site, float p) -> Tensor", _dropout_bwd, _dropout_bwd_fake)


# ---------------------------------------------------------------------------------------------- fused feed-forward block
def _ln_mlp_fwd(x: Tensor, gamma: Tensor, beta: Tensor, w1: Tensor, b1: Tensor, w2: Tensor, b2: Tensor,
                eps: float = 1e-5) -> Tensor:
    return ops.ln_mlp_fwd(x.contiguous(), gamma, beta, w1.contiguous(), b1, w2.contiguous(), b2, eps=eps)


def _ln_mlp_fwd_fake(x, gamma, beta, w1, b1, w2, b2, eps=1e-5):
    torch._check(x.dim() == 2 and w1.shape == (w1.shape[0], x.shape[1]) and w2.shape == (x.shape[1], w1.shape[0]),
                 lambda: "ln_mlp_fwd: x [M, D], w1 [H, D], w2 [D, H]")
    return x.new_empty(x.shape)


_define("ln_mlp_fwd(Tensor x, Tensor gamma, Tensor beta, Tensor w1, Tensor b1, Tensor w2, Tensor b2, float eps=1e-5) -> Tensor",
        _ln_mlp_fwd, _ln_mlp_fwd_fake)


# ---------------------------------------------------------------------------------------------- mask sampling
def _mask_indices(noise: Tensor, offsets: List[int], lengths: List[int], n_masked: List[int]) -> Tuple[Tensor, Tensor]:
    segs = list(zip(offsets, lengths, n_masked))
    masked, unmasked, _ = ops.mask_indices(noise.contiguous(), segs, want_slots=True)
    return masked, unmasked


def _mask_indices_fake(noise, offsets, lengths, n_masked):
    torch._check(noise.dim() == 2 and noise.dtype == torch.float32, lambda: "mask_indices: noise fp32 [B, n]")
    torch._check(len(offsets) == len(lengths) == len(n_masked), lambda: "mask_indices: ragged segment lists")
    nm = sum(n_masked)
    nu = sum(lengths) - nm
    return (noise.new_empty((noise.shape[0], nm), dtype=torch.int64), noise.new_empty((noise.shape[0], nu), dtype=torch.int64))


_define("mask_indices(Tensor noise, int[] offsets, int[] lengths, int[] n_masked) -> (Tensor, Tensor)",
        _mask_indices, _mask_indices_fake)


# ---------------------------------------------------------------------------------------------- patchify + LayerNorm
def _patch_layernorm(maps: List[Tensor], patch_h: int, patch_w: int, token_base: int, tok_idx: Optional[Tensor], col0: int,
                     ncols: int, gamma: Tensor, beta: Tensor, eps: float = 1e-5) -> Tensor:
    ps = ops.make_patch_source([m.contiguous() for m in maps], patch_h, patch_w, token_base)
    out, _ = ops.patch_layernorm(ps, maps[0].shape[0], ncols, gamma, beta, tok_idx=tok_idx, col0=col0, want_xhat=False, eps=eps)
    return out


def _patch_layernorm_fake(maps, patch_h, patch_w, token_base, tok_idx, col0, ncols, gamma, beta, eps=1e-5):
    B, Cc = maps[0].shape[0], maps[0].shape[1]
    return maps[0].new_empty((B * ncols, patch_h * patch_w * Cc), dtype=torch.bfloat16)


_define("patch_layernorm(Tensor[] maps, int patch_h, int patch_w, int token_base, Tensor? tok_idx, int col0, int ncols, "
        "Tensor gamma, Tensor beta, float eps=1e-5) -> Tensor", _patch_layernorm, _patch_layernorm_fake)


# ---------------------------------------------------------------------------------------------- masked-patch MSE
def _masked_patch_mse(maps: List[Tensor], patch_h: int, patch_w: int, token_base: int, tok_idx: Optional[Tensor], col0: int,
                      ncols: int, pred: Tensor, weight: float = 1.0) -> Tuple[Tensor, Tensor]:
    ps = ops.make_patch_source([m.contiguous() for m in maps], patch_h, patch_w, token_base)
    loss = torch.zeros(1, dtype=torch.float32, device=pred.device)
    dpred = ops.mse_loss(ps, maps[0].shape[0], ncols, pred.contiguous(), weight / pred.numel(), loss, tok_idx=tok_idx, col0=col0)
    return loss.reshape(()), dpred


def _masked_patch_mse_fake(maps, patch_h, patch_w, token_base, tok_idx, col0, ncols, pred, weight=1.0):
    return pred.new_empty((), dtype=torch.float32), pred.new_empty(pred.shape, dtype=torch.bfloat16)


_define("masked_patch_mse(Tensor[] maps, int patch_h, int patch_w, int token_base, Tensor? tok_idx, int col0, int ncols, "
        "Tensor pred, float weight=1.0) -> (Tensor, Tensor)", _masked_patch_mse, _masked_patch_mse_fake)


# ---------------------------------------------------------------------------------------------- vt_load
def _vt_load_image(image: Tensor, frame_stack: int, lo: float = 0.0, hi: float = 1.0) -> Tensor:
    from .data import _image_view
    return _image_view(image.contiguous(), frame_stack, lo, hi).materialize()


def _vt_load_image_fake(image, frame_stack, lo=0.0, hi=1.0):
    if image.dim() == 5:
        B, F, H, W, _ = image.shape
        return image.new_empty((B, 3 * F, H, W), dtype=torch.float32)
    B, H, W, Cc = image.shape
    return image.new_empty((B, Cc, H, W), dtype=torch.float32)


_define("vt_load_image(Tensor image, int frame_stack, float lo=0.0, float hi=1.0) -> Tensor", _vt_load_image, _vt_load_image_fake)


def _vt_load_tactile(tactile: Tensor, frame_stack: int, sensor: int, lo: float = -1.0, hi: float = 1.0) -> Tensor:
    from .data import _tactile_views
    return _tactile_views(tactile.contiguous(), frame_stack, lo, hi)[f"tactile{sensor + 1}"].materialize()


def _vt_load_tactile_fake(tactile, frame_stack, sensor, lo=-1.0, hi=1.0):
    return tactile.new_empty((tactile.shape[0], 3 * frame_stack, tactile.shape[-2], tactile.shape[-1]), dtype=torch.float32)


_define("vt_load_tactile(Tensor tactile, int frame_stack, int sensor, float lo=-1.0, float hi=1.0) -> Tensor",
        _vt_load_tactile, _vt_load_tactile_fake)
