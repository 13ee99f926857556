"""Drop-in for the DINO-side encoder `models/VTT.py::VTT` of the reference (SURVEY.md §8 row a-16;
/root/reference/models/VTT.py:77-426): same keyword-only constructor, parameter / buffer names
(`image_to_patch_embedding.{1,2,3}`, `tactile_to_patch_embedding_{1,2}.{1,2,3}`, `pos_embedding`,
`register_tokens`, `transformer.*`, `norm.*`, `pos_embed.frequency_bands`), timm-style init, and the
`forward_features(x, masks) -> dict` / `forward` outputs, computing through the sm_100a kernels:

    from m3l_b200.vtt import VTT            # instead of: from models.VTT import VTT

Kernel sequence (all through the C-ABI, no CPU path): per modality and keep-index list, the fused
patchify + gather + LayerNorm(P) kernel (only the kept tokens are embedded — LN/Linear/LN is per token,
so this equals the reference's embed-all-then-gather), the tcgen05 GEMM, LayerNorm(D) fused with the
sinusoidal position add and the scatter into the (mask, sample, token) row order; then the shared
transformer stack and the final LayerNorm(eps=1e-6).  Register-token rows are a plain copy.
"""
from __future__ import annotations

import math
from functools import partial
from typing import List, Optional

import torch
from torch import nn
from torch.nn.init import trunc_normal_

from . import engine, ops
from ._lib import M3LError
from .arena import ParamArena
from .vtmae import Patchify, Transformer, pair


class SinusoidalEmbed(nn.Module):
    """tactile_ssl/model/layers/patch_embed.py:133-213 — table over the integer patch grid, per axis
    cat[sin(c * bands), cos(c * bands)], bands = 10000^(-linspace(0, 1, nb + 1)[:-1]), truncated to embed_dim;
    cached on first use."""

    def __init__(self, size, stride, embed_dim=768):
        super().__init__()
        size, stride = list(size), list(stride)
        assert len(size) < 4, "Sinusoidal position embeddings only support 1D, 2D and 3D grids."
        assert len(size) == len(stride), "size and stride must have the same length"
        self.patches_resolution = [s // stride[i] for i, s in enumerate(size)]
        self.embed_dim = embed_dim
        self.num_patches = int(math.prod(self.patches_resolution))
        assert embed_dim % 2 == 0, "Embedding dimension must be divisible by 2"
        self.num_bands = math.ceil(embed_dim / (2 * len(size)))
        bands = torch.stack([torch.linspace(0, 1.0, steps=self.num_bands + 1)[:-1] for _ in size], dim=0)
        self.register_buffer("frequency_bands", 10000 ** -bands)
        self.register_buffer("cached_encoding", None, persistent=False)

    def forward(self, device, normalized_coords: bool = False):
        if self.cached_encoding is not None:
            return self.cached_encoding if self.cached_encoding.device == device else self.cached_encoding.to(device)
        axes = [torch.arange(0, r, dtype=torch.float, device=device) for r in self.patches_resolution]
        grid = torch.stack(torch.meshgrid(*axes, indexing="ij"), dim=-1).reshape(-1, len(axes))
        feat = grid[..., None] * self.frequency_bands.to(device)
        enc = torch.cat([torch.sin(feat), torch.cos(feat)], dim=-1).flatten(-2, -1)
        self.cached_encoding = enc[..., : self.embed_dim]
        return self.cached_encoding


def _patch_embedding(patch_h, patch_w, patch_dim, dim):
    return nn.Sequential(Patchify(patch_h, patch_w), nn.LayerNorm(patch_dim), nn.Linear(patch_dim, dim), nn.LayerNorm(dim))


_EMBEDS = ("image_to_patch_embedding", "tactile_to_patch_embedding_1", "tactile_to_patch_embedding_2")
_KEYS = ("image", "tactile1", "tactile2")


class VTT(nn.Module):
    def __init__(self, *, image_size, tactile_size, image_patch_size, tactile_patch_size, dim, depth, heads, mlp_dim,
                 image_channels=3, tactile_channels=3, dim_head=64, dropout=0., emb_dropout=0, num_tactiles=2,
                 frame_stack=1, pos_embed_fn="sinusoidal", num_register_tokens: int = 0, num_frames: int = 1):
        super().__init__()
        image_height, image_width = pair(image_size)
        tactile_height, tactile_width = pair(tactile_size)
        iph, ipw = pair(image_patch_size)
        tph, tpw = pair(tactile_patch_size)
        self.image_height, self.image_width = image_height, image_width
        self.tactile_height, self.tactile_width = tactile_height, tactile_width
        self.image_patch_height, self.image_patch_width = iph, ipw
        self.tactile_patch_height, self.tactile_patch_width = tph, tpw
        self.image_channels, self.tactile_channels = image_channels, tactile_channels
        self.frame_stack = frame_stack
        assert image_height % iph == 0 and image_width % ipw == 0, 'Image dimensions must be divisible by the patch size.'
        assert tactile_height % tph == 0 and tactile_width % tpw == 0, 'Tactile dimensions must be divisible by the patch size.'
        self.num_patches_image = (image_height // iph) * (image_width // ipw)
        self.num_patches_tactile = (tactile_height // tph) * (tactile_width // tpw) * num_tactiles
        self.num_patches = self.num_patches_image + self.num_patches_tactile
        self.image_to_patch_embedding = _patch_embedding(iph, ipw, image_channels * iph * ipw, dim)
        self.tactile_to_patch_embedding_1 = _patch_embedding(tph, tpw, tactile_channels * tph * tpw, dim)
        self.tactile_to_patch_embedding_2 = _patch_embedding(tph, tpw, tactile_channels * tph * tpw, dim)
        self.pos_embedding = nn.Parameter(torch.randn(1, self.num_patches + 1, dim))
        self.dropout = nn.Dropout(emb_dropout)
        self.transformer = Transformer(dim, depth, heads, dim_head, mlp_dim, dropout)
        self.to_latent = nn.Identity()
        assert num_register_tokens >= 0
        self.num_register_tokens = num_register_tokens
        self.register_tokens = nn.Parameter(torch.zeros(1, num_register_tokens, dim)) if num_register_tokens else None
        self.pos_embed_fn = pos_embed_fn
        self.num_frames = num_frames
        self.embed_dim = dim
        if pos_embed_fn != "sinusoidal":
            # the reference builds no table for "learned" and fails on first use (models/VTT.py:201-205,237)
            raise NotImplementedError("Unknown position embedding function")
        self.pos_embed = SinusoidalEmbed([image_height * 3, image_width], [image_patch_size, image_patch_size], embed_dim=dim)
        self.norm = partial(nn.LayerNorm, eps=1e-6)(dim)
        self.head = nn.Identity()
        self.init_weights()
        self._arena: Optional[ParamArena] = None

    def init_weights(self):
        """models/VTT.py:222-228,801-809: trunc_normal_(std=0.02) Linear weights, zero biases, LN (1, 0)."""
        if self.register_tokens is not None:
            nn.init.normal_(self.register_tokens, std=1e-6)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                trunc_normal_(m.weight, std=0.02)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)
            elif isinstance(m, nn.LayerNorm):
                nn.init.zeros_(m.bias)
                nn.init.ones_(m.weight)

    def interpolate_pos_encoding(self, img_shape, img_dtype, device):
        return self.pos_embed(device).float().unsqueeze(0)

    # ------------------------------------------------------------------------------------------
    def _own_arena(self) -> ParamArena:
        dev = self.norm.weight.device
        if dev.type != "cuda":
            raise M3LError("m3l_b200.vtt.VTT needs CUDA parameters (there is no CPU fallback)")
        if self._arena is None or self._arena.device != dev:
            named = [(k, p) for k, p in self.named_parameters() if k != "pos_embedding"]
            self._arena = ParamArena(named, dev)
        self._arena.sync()
        return self._arena

    def forward_features(self, x, masks: Optional[List[torch.Tensor]] = None):
        """x: dict(image (B,C,H,W), tactile1, tactile2) fp32 CUDA; masks: list of (B, K) keep-index tensors shared
        by the three modalities (tactile_ssl/utils/__init__.py:25-36) -> the reference's dict of (len(masks)*B, ., D)."""
        A = self._own_arena()
        maps = []
        for k in _KEYS:
            v = x[k]
            if v.device != A.device:
                raise M3LError(f"input '{k}' is on {v.device}, the module on {A.device} (no CPU path)")
            maps.append(v.detach().to(torch.float32).contiguous())
        n_per = self.num_patches_image
        if not (maps[1].shape[2] // self.tactile_patch_height) * (maps[1].shape[3] // self.tactile_patch_width) == n_per:
            raise M3LError("models/VTT.py::VTT slices ONE position table over the three maps (:290-292): image and "
                           "tactile maps must have the same patch count")
        if masks is not None:
            masks = [m.to(device=A.device, dtype=torch.int64).contiguous() for m in masks]
        names = list(A.names)
        xn, xpre = _VTTFn.apply(self, A, maps, masks, tuple(names), *[A.params[n] for n in names])
        R = self.num_register_tokens
        return {"x_norm_regtokens": xn[:, :R], "x_norm_patchtokens": xn[:, R:], "x_prenorm": xpre, "masks": masks}

    def forward(self, *args, **kwargs):
        return self.forward_features(*args, **kwargs)["x_norm_patchtokens"]


class _VTTFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, A, maps, masks, names, *params):
        dev = A.device
        need = any(ctx.needs_input_grad)
        B = maps[0].shape[0]
        D, R, n_per = mod.embed_dim, mod.num_register_tokens, mod.num_patches_image
        P = len(masks) if masks is not None else 1
        K = masks[0].shape[1] if masks is not None else n_per
        n, Beff = R + 3 * K, P * B
        pos = mod.pos_embed(dev).float().contiguous()
        x0 = torch.empty((Beff * n, D), dtype=torch.bfloat16, device=dev)
        b = torch.arange(B, device=dev)[:, None]
        j = torch.arange(K, device=dev)[None]
        sizes = [(mod.image_patch_height, mod.image_patch_width)] + [(mod.tactile_patch_height, mod.tactile_patch_width)] * 2
        emb_saved = []
        for m, (pre, (ph, pw)) in enumerate(zip(_EMBEDS, sizes)):
            ps = ops.make_patch_source([maps[m]], ph, pw, 0)
            for p in range(P):
                mk = masks[p] if masks is not None else None
                a, xhat = ops.patch_layernorm(ps, B, K, A.f32(pre + ".1.weight"), A.f32(pre + ".1.bias"), tok_idx=mk,
                                              col0=0, want_xhat=need)
                e = ops.gemm(a, A.bf(pre + ".2.weight"), bias=A.f32(pre + ".2.bias"), out_dtype=torch.float32)
                dst = ((p * B + b) * n + R + m * K + j).reshape(-1).to(torch.int32)
                tok = mk if mk is not None else j.expand(B, K)
                pos_row = (m * n_per + tok).reshape(-1).to(torch.int32)
                _, st = ops.layernorm_fwd(e, A.f32(pre + ".3.weight"), A.f32(pre + ".3.bias"), out=x0, dst_row=dst,
                                          add1=pos, add1_row=pos_row, want_stats=need)
                if need:
                    emb_saved.append((pre, a, xhat, e, st, dst))
        if R:
            x0.view(Beff, n, D)[:, :R] = A.bf("register_tokens")
        tr = mod.transformer
        spec = engine.StackSpec("transformer", tr.dim, tr.depth, tr.heads, tr.dim_head, tr.mlp_dim)
        saved = [] if need else None
        xe = engine.stack_fwd(A, spec, x0, Beff, n, saved, p_drop=engine.p_drop(tr))
        xt, st_t = ops.layernorm_fwd(xe, A.f32("transformer.norm.weight"), A.f32("transformer.norm.bias"), want_stats=need)
        xn, st_n = ops.layernorm_fwd(xt, A.f32("norm.weight"), A.f32("norm.bias"), want_stats=need, eps=1e-6)
        ctx.c = (A, spec, emb_saved, saved, xe, st_t, xt, st_n, Beff, n, D, R, names)
        return xn.float().reshape(Beff, n, D), xt.float().reshape(Beff, n, D)

    @staticmethod
    def backward(ctx, g_norm, g_pre):
        A, spec, emb_saved, saved, xe, st_t, xt, st_n, Beff, n, D, R, names = ctx.c
        gflat = A.new_grad_buffer()
        G = engine.GradView(A, gflat)
        dn = g_norm.reshape(Beff * n, D).to(torch.bfloat16).contiguous()
        skip = g_pre.reshape(Beff * n, D).to(torch.bfloat16).contiguous()
        dxt = ops.layernorm_bwd(dn, xt, st_n, A.f32("norm.weight"), dgamma=G("norm.weight"), dbeta=G("norm.bias"), skip=skip)
        dxe = ops.layernorm_bwd(dxt, xe, st_t, A.f32("transformer.norm.weight"), dgamma=G("transformer.norm.weight"),
                                dbeta=G("transformer.norm.bias"),
                                dx_colsum=engine.stack_dx_colsum(G, spec, saved))
        dx0 = engine.stack_bwd(A, G, spec, dxe, Beff, n, saved)
        if R:
            G("register_tokens").copy_(dx0.view(Beff, n, D)[:, :R].float().sum(0, keepdim=True))
        for pre, a, xhat, e, st, dst in emb_saved:
            de = ops.layernorm_bwd(dx0, e, st, A.f32(pre + ".3.weight"), dgamma=G(pre + ".3.weight"),
                                   dbeta=G(pre + ".3.bias"), src_row=dst)
            ops.colsum(de, G(pre + ".2.bias"))
            engine.wgrad(de, a, G(pre + ".2.weight"))
            da = ops.gemm(de, A.bf_t(pre + ".2.weight"))
            ops.ln_param_grad(da, xhat, G(pre + ".1.weight"), G(pre + ".1.bias"))
        return (None, None, None, None, None, *[A.view(gflat, k) for k in names])
