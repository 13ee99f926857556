"""Test helper: the dropout masks of csrc/dropout.cuh regenerated in numpy, and the oracle transformer with a hook
that applies them.

Mask definition (include/m3l_b200.h): Philox4x32-10 under the 64-bit key, counter (col >> 3, row, plane, site); the
four output words are eight 16-bit uniforms, low half first; element `col & 7` is kept iff its uniform is
>= thr = floor(p * 65536 + 0.5) and is then multiplied by float32(65536 / (65536 - thr)).
"""
from __future__ import annotations

import contextlib
import math

import numpy as np
import torch

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: uint32 array [..., 4]; key: (k0, k1) ints.  Returns uint32 [..., 4]."""
    c = [np.asarray(ctr, dtype=np.uint64)[..., i] for i in range(4)]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for r in range(10):
        if r:
            k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
        p0, p1 = _M0 * c[0], _M1 * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & _MASK32, p1 >> np.uint64(32), p1 & _MASK32
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
    return np.stack(c, -1).astype(np.uint32)


def threshold(p: float):
    thr = int(math.floor(np.float32(p) * np.float64(65536.0) + 0.5))
    return thr, np.float32(65536.0 / (65536.0 - thr))


def uniforms(key: int, site: int, rows: int, cols: int, plane: int = 0) -> np.ndarray:
    """uint16-valued int64 array [rows, cols] of the uniforms of (row, col) at this plane and site."""
    groups = (cols + 7) // 8
    r, g = np.meshgrid(np.arange(rows, dtype=np.uint64), np.arange(groups, dtype=np.uint64), indexing="ij")
    ctr = np.stack([g, r, np.full_like(r, plane), np.full_like(r, site)], -1)
    w = philox4x32_10(ctr, (key & 0xFFFFFFFF, (key >> 32) & 0xFFFFFFFF)).astype(np.int64)   # [rows, groups, 4]
    u = np.stack([w & 0xFFFF, w >> 16], -1).reshape(rows, groups * 8)                      # word 0 low, high, ...
    return u[:, :cols]


def mask(key: int, site: int, rows: int, cols: int, p: float, plane: int = 0) -> np.ndarray:
    """float32 [rows, cols]: 0 where dropped, the scale where kept."""
    thr, scale = threshold(p)
    return np.where(uniforms(key, site, rows, cols, plane) >= thr, scale, np.float32(0)).astype(np.float32)


def attn_mask(key: int, site: int, B: int, H: int, n: int, p: float) -> np.ndarray:
    """float32 [B, H, n (query), n (key)]."""
    return np.stack([np.stack([mask(key, site, n, n, p, plane=b * H + h) for h in range(H)]) for b in range(B)])


class MaskHook:
    """drop hook (layer, site, tensor) -> tensor of the oracle transformer: multiplies by the numpy masks of one key,
    with the row layout of the kernels (activations [B*n, features], attention planes b * heads + h)."""

    def __init__(self, key: int, p: float):
        self.key, self.p = key, p

    def z(self, layer: int, s: int, t: torch.Tensor) -> torch.Tensor:
        site = (layer << 2) | s
        if s == 0:
            B, H, n, _ = t.shape
            z = attn_mask(self.key, site, B, H, n, self.p)
        else:
            z = mask(self.key, site, t.shape[0] * t.shape[1], t.shape[2], self.p).reshape(t.shape)
        return torch.from_numpy(z).to(device=t.device, dtype=t.dtype)

    def __call__(self, layer: int, s: int, t: torch.Tensor) -> torch.Tensor:
        return t * self.z(layer, s, t)


def transformer(x, sd, prefix, depth, heads, dim_head, drop=None):
    """oracle.vtmae_oracle.transformer with vit_pytorch's four Dropout sites routed through drop(layer, site, t)."""
    import torch.nn.functional as F
    from oracle.vtmae_oracle import layer_norm, linear
    d = drop if drop is not None else (lambda l, s, t: t)
    b, n, _ = x.shape
    scale = dim_head ** -0.5
    for l in range(depth):
        pa, pf = f"{prefix}.layers.{l}.0", f"{prefix}.layers.{l}.1"
        h = layer_norm(x, sd, pa + ".norm")
        q, k, v = F.linear(h, sd[pa + ".to_qkv.weight"]).chunk(3, dim=-1)
        q, k, v = (t.reshape(b, n, heads, dim_head).transpose(1, 2) for t in (q, k, v))
        attn = d(l, 0, torch.softmax(torch.matmul(q, k.transpose(-1, -2)) * scale, dim=-1))
        o = torch.matmul(attn, v).transpose(1, 2).reshape(b, n, heads * dim_head)
        if (pa + ".to_out.0.weight") in sd:
            o = d(l, 1, linear(o, sd, pa + ".to_out.0"))
        x = o + x
        h = layer_norm(x, sd, pf + ".net.0")
        h = d(l, 2, F.gelu(linear(h, sd, pf + ".net.1")))
        x = d(l, 3, linear(h, sd, pf + ".net.4")) + x
    return layer_norm(x, sd, prefix + ".norm")


@contextlib.contextmanager
def oracle_dropout(hooks: dict):
    """Within the block, the oracle's transformers (oracle.vtmae_oracle / vtt_dino_oracle) apply drop hooks:
    hooks maps a parameter prefix ("encoder.transformer", "transformer", ...) to a hook, or to a list of hooks used
    by successive calls with that prefix."""
    from oracle import vtmae_oracle, vtt_dino_oracle
    calls = {}

    def patched(x, sd, prefix, depth, heads, dim_head):
        h = hooks.get(prefix)
        if isinstance(h, list):
            i = calls.get(prefix, 0)
            calls[prefix] = i + 1
            h = h[i]
        return transformer(x, sd, prefix, depth, heads, dim_head, drop=h)

    saved = vtmae_oracle.transformer, vtt_dino_oracle.transformer
    vtmae_oracle.transformer = vtt_dino_oracle.transformer = patched
    try:
        yield
    finally:
        vtmae_oracle.transformer, vtt_dino_oracle.transformer = saved
