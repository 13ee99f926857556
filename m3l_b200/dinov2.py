"""Frozen DINOv2 ViT-S/14-with-registers image branch of the DINO-tac-MAE variant, on the kernel path, and the
feature extractor that concatenates its class token with the MAE latents.

Reference (paths under /root/reference):
  train_dino_tac_mae.py:29-31                       dino = torch.hub.load('facebookresearch/dinov2', 'dinov2_vits14_reg'); frozen
  models/pretrain_models_dino_cat_mae.py:792-841    MAEExtractor(observation_space, dino_model, mae_model, dim_embeddings, ...)
  models/pretrain_models_dino_cat_mae.py:866-904    forward: MAE latents -> vit_layer -> token mean, DINO class token of the
                                                    mid frame, cat, 3-layer mlp

`DinoV2` has the torch.hub model's constructor defaults, module tree and state_dict names, so
`DinoV2().load_state_dict(hub_model.state_dict())` works; its forward (no gradients: the reference freezes it) is a
sequence of the C-ABI kernels: patchify (raw observation or NCHW map) -> tcgen05 GEMM (patch embedding as a Linear over
(p1, p2, c)-ordered patches) -> token assembly (class / register tokens + position table) -> 12 x [LayerNorm, QKV GEMM,
fused attention (6 heads x 64), projection GEMM with LayerScale folded into its weights + residual, LayerNorm, FF1 GEMM +
GELU, FF2 GEMM (LayerScale folded) + residual] -> final LayerNorm of the class rows only.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F
from torch import nn

from . import engine, ops
from ._lib import M3LError
from .data import RawMap, vt_load_lazy


class _LayerScale(nn.Module):
    def __init__(self, dim, init_values=1.0):
        super().__init__()
        self.gamma = nn.Parameter(init_values * torch.ones(dim))


class _Attention(nn.Module):
    def __init__(self, dim, num_heads):
        super().__init__()
        self.num_heads = num_heads
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.proj = nn.Linear(dim, dim, bias=True)


class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio, init_values):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = _Attention(dim, num_heads)
        self.ls1 = _LayerScale(dim, init_values)
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))
        self.ls2 = _LayerScale(dim, init_values)


class _PatchEmbed(nn.Module):
    def __init__(self, patch_size, embed_dim):
        super().__init__()
        self.proj = nn.Conv2d(3, embed_dim, kernel_size=patch_size, stride=patch_size)


class DinoV2(nn.Module):
    """dinov2_vits14_reg by default (embed_dim 384, depth 12, 6 heads, 4 register tokens, 37 x 37 position grid)."""

    def __init__(self, img_size=518, patch_size=14, embed_dim=384, depth=12, num_heads=6, mlp_ratio=4, num_register_tokens=4,
                 init_values=1.0):
        super().__init__()
        if embed_dim // num_heads != 64:
            raise M3LError("m3l_b200.DinoV2: the fused attention kernel is built for 64-wide heads")
        self.patch_size, self.embed_dim, self.num_heads = patch_size, embed_dim, num_heads
        self.num_register_tokens = num_register_tokens
        g = img_size // patch_size
        self.patch_embed = _PatchEmbed(patch_size, embed_dim)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, 1 + g * g, embed_dim))
        self.register_tokens = nn.Parameter(torch.zeros(1, num_register_tokens, embed_dim))
        self.mask_token = nn.Parameter(torch.zeros(1, embed_dim))
        self.blocks = nn.ModuleList([_Block(embed_dim, num_heads, mlp_ratio, init_values) for _ in range(depth)])
        self.norm = nn.LayerNorm(embed_dim, eps=1e-6)
        nn.init.trunc_normal_(self.pos_embed, std=0.02)
        nn.init.normal_(self.cls_token, std=1e-6)
        nn.init.normal_(self.register_tokens, std=1e-6)
        self._prep: Optional[dict] = None

    # ------------------------------------------------------------------ frozen-weight preparation
    def _version(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _pos_table(self, gh, gw):
        pe = self.pos_embed.detach().float()
        n_pos = pe.shape[1] - 1
        if not (n_pos == gh * gw and gh == gw):
            g = int(math.sqrt(n_pos))
            D = pe.shape[-1]
            patch = pe[:, 1:].reshape(1, g, g, D).permute(0, 3, 1, 2)
            patch = F.interpolate(patch, size=(gh, gw), mode="bicubic", align_corners=False, antialias=True)
            pe = torch.cat([pe[:, :1], patch.permute(0, 2, 3, 1).reshape(1, gh * gw, D)], 1)
        return pe[0]

    def _prepare(self, gh, gw):
        """bf16 GEMM operands and the additive token table (computed once per weight version and input grid; the
        network is frozen, so this is load-time work): conv weight re-ordered to the (p1, p2, c) patch order and
        K-padded to a multiple of 8; LayerScale folded into the projection / FF2 weights and biases."""
        key = (self._version(), gh, gw)
        if self._prep is not None and self._prep["key"] == key:
            return self._prep
        dev = self.cls_token.device
        if dev.type != "cuda":
            raise M3LError("m3l_b200.DinoV2 needs its parameters on a CUDA device (no CPU fallback)")
        D, R, ps = self.embed_dim, self.num_register_tokens, self.patch_size
        f32 = lambda t: t.detach().to(device=dev, dtype=torch.float32).contiguous()
        bf = lambda t: t.detach().to(device=dev, dtype=torch.float32).to(torch.bfloat16).contiguous()
        P = 3 * ps * ps
        ld = (P + 7) // 8 * 8
        w = self.patch_embed.proj.weight.detach().float().permute(0, 2, 3, 1).reshape(D, P)      # (ky, kx, c) order
        wpe = torch.zeros(D, ld, device=dev)
        wpe[:, :P] = w
        pos = self._pos_table(gh, gw)
        add1 = torch.cat([self.cls_token.detach().float()[0] + pos[:1], self.register_tokens.detach().float()[0], pos[1:]], 0)
        prep = {"key": key, "ld": ld, "wpe": wpe.to(torch.bfloat16).contiguous(), "bpe": f32(self.patch_embed.proj.bias),
                "add1": f32(add1), "zero": torch.zeros(D, device=dev), "norm": (f32(self.norm.weight), f32(self.norm.bias)),
                "blocks": [], "slots": {}, "cls_rows": {}}
        for b in self.blocks:
            g1, g2 = b.ls1.gamma.detach().float(), b.ls2.gamma.detach().float()
            prep["blocks"].append(dict(
                n1=(f32(b.norm1.weight), f32(b.norm1.bias)), n2=(f32(b.norm2.weight), f32(b.norm2.bias)),
                wqkv=bf(b.attn.qkv.weight), bqkv=f32(b.attn.qkv.bias),
                wproj=bf(g1[:, None] * b.attn.proj.weight.detach().float()), bproj=f32(g1 * b.attn.proj.bias.detach().float()),
                w1=bf(b.mlp.fc1.weight), b1=f32(b.mlp.fc1.bias),
                w2=bf(g2[:, None] * b.mlp.fc2.weight.detach().float()), b2=f32(g2 * b.mlp.fc2.bias.detach().float())))
        self._prep = prep
        return prep

    # ------------------------------------------------------------------ forward
    use_cuda_graph = True        # replay the ~90-kernel forward from a CUDA graph cached per input shape

    @torch.no_grad()
    def forward(self, x, return_tokens: bool = False):
        """x: fp32 (B, 3, H, W) CUDA tensor, or a data.RawMap view of three channels of a raw observation.
        Returns the normalised class token (B, embed_dim) fp32 (what the hub model's forward returns).
        The network is frozen and the call is launch-bound at rollout / small-minibatch sizes (7 kernels per block behind
        Python + ctypes), so the kernel sequence is captured once per (batch, height, width) and replayed: the three input
        channels are first gathered into a static NCHW buffer (one `m3l_vt_load` launch, or a copy for tensor inputs)."""
        if not self.use_cuda_graph or return_tokens or torch.cuda.is_current_stream_capturing():
            return self._forward_eager(x, return_tokens)
        B, C, H, W = x.shape
        prep = self._prepare(H // self.patch_size, W // self.patch_size)
        cache = prep.setdefault("graphs", {})
        ent = cache.get((B, H, W))
        dev = prep["wpe"].device
        if ent is None:
            if len(cache) >= 4:
                cache.pop(next(iter(cache)))
            static_in = torch.zeros((B, 3, H, W), dtype=torch.float32, device=dev)
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._forward_eager(static_in, False)          # warm-up: lazy tables, kernel attributes, allocator
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with engine.capture_guard(), torch.cuda.graph(g):
                out = self._forward_eager(static_in, False)
            ent = cache[(B, H, W)] = (g, static_in, out)
        g, static_in, out = ent
        if isinstance(x, RawMap):
            ops.vt_load_map(x, out=static_in)
        else:
            if not x.is_cuda:
                raise M3LError("m3l_b200.DinoV2: input is not on a CUDA device (no CPU fallback)")
            static_in.copy_(x, non_blocking=True)
        g.replay()
        return out.clone()

    @torch.no_grad()
    def _forward_eager(self, x, return_tokens: bool = False):
        if not isinstance(x, RawMap):
            if not x.is_cuda:
                raise M3LError("m3l_b200.DinoV2: input is not on a CUDA device (no CPU fallback)")
            x = x.detach().to(torch.float32)
            B, C, H, W = x.shape
            # any strided NCHW view (e.g. a channel slice of the stacked image) is a layout-1 source with identity
            # normalisation: no copy
            x = RawMap(x, (B, C, H, W), 0, x.stride(0), C, 0, x.stride(1), x.stride(2), x.stride(3), 0.0, 1.0,
                       strided_view=True)
        B, C, H, W = x.shape
        assert C == 3, "DINOv2 takes three image channels"
        ps, D, R, heads = self.patch_size, self.embed_dim, self.num_register_tokens, self.num_heads
        gh, gw = H // ps, W // ps
        npatch, n = gh * gw, 1 + R + gh * gw
        prep = self._prepare(gh, gw)
        dev = prep["wpe"].device
        slots = prep["slots"].get(B)
        if slots is None:
            t = torch.arange(n, device=dev, dtype=torch.int32) - (1 + R)
            slots = prep["slots"][B] = torch.where(t >= 0, t, torch.full_like(t, -1)).repeat(B).contiguous()
            r = torch.arange(B * n, device=dev, dtype=torch.int32)
            prep["cls_rows"][B] = torch.where(r % n == 0, r // n, torch.full_like(r, -1)).contiguous()
        src = ops.make_patch_source([x], ps, ps, 0)
        cols = ops.patchify(src, B, npatch, ld=prep["ld"])
        tok = ops.gemm(cols, prep["wpe"], bias=prep["bpe"])
        xs = ops.decoder_assemble_fwd(tok, npatch, prep["zero"], slots, B, n, add1=prep["add1"])
        scale = 64 ** -0.5
        for blk in prep["blocks"]:
            y, _ = ops.layernorm_fwd(xs, *blk["n1"], eps=1e-6, want_stats=False)
            qkv = ops.gemm(y, blk["wqkv"], bias=blk["bqkv"])
            o, _ = ops.mha_fwd(qkv, B, n, heads, 64, scale)
            xs = ops.gemm(o, blk["wproj"], bias=blk["bproj"], residual=xs)
            y, _ = ops.layernorm_fwd(xs, *blk["n2"], eps=1e-6, want_stats=False)
            h = ops.gemm(y, blk["w1"], bias=blk["b1"], act=ops.GELU_FWD)
            xs = ops.gemm(h, blk["w2"], bias=blk["b2"], residual=xs)
        if return_tokens:
            out, _ = ops.layernorm_fwd(xs, *prep["norm"], eps=1e-6, want_stats=False)
            return out.float().reshape(B, n, D)
        cls, _ = ops.layernorm_fwd(xs, *prep["norm"], eps=1e-6, want_stats=False, out_rows=B, dst_row=prep["cls_rows"][B])
        return cls.float()


def mid_frame_view(image, frame_stack: int):
    """The three channels [3*mid-3, 3*mid), mid = frame_stack // 2, of the model's image input
    (pretrain_models_dino_cat_mae.py:884-889) as something DinoV2.forward reads without a copy."""
    mid = frame_stack // 2
    c0 = 3 * mid - 3
    if isinstance(image, RawMap):
        assert image.cg == 3, "mid-frame selection needs frame-grouped channels"
        B, _, H, W = image.shape
        return RawMap(image.t, (B, 3, H, W), image.offset + (c0 // 3) * image.sf, image.sb, 3, 0, image.sch, image.sy,
                      image.sx, image.lo, image.span)
    return image[:, c0:c0 + 3]


# --------------------------------------------------------------------------------------------
# DINO-cat-MAE feature extractor (models/pretrain_models_dino_cat_mae.py:792-904)
# --------------------------------------------------------------------------------------------
from .vtmae import MAEExtractor as _MAEExtractorBase, VTT as _VTT      # noqa: E402


class DinoCatMAEExtractor(_MAEExtractorBase):
    """`MAEExtractor` of models/pretrain_models_dino_cat_mae.py: same constructor argument order
    (observation_space, dino_model, mae_model, dim_embeddings, vision_only_control, frame_stack), same attributes
    (`vit_layer` at 70 x 70 / patch 14, `mlp`, `query`, `query_projection`, `key_projection`), output (B, dim_embeddings).
    The MAE chain (encoder over all tokens, extra block, token mean) and the frozen DINOv2 forward run on the kernel
    path and read the raw observations in place; the small trainable policy-side `mlp` on the (B, 2*dim) concatenation
    stays an ordinary autograd nn.Sequential, as in the reference."""

    def __init__(self, observation_space, dino_model, mae_model, dim_embeddings, vision_only_control, frame_stack) -> None:
        super().__init__(observation_space, mae_model, dim_embeddings, vision_only_control, frame_stack)
        self.dino_model = dino_model
        self.vit_layer = _VTT(image_size=(70, 70), tactile_size=(70, 70), image_patch_size=14, tactile_patch_size=14,
                              dim=dim_embeddings, depth=1, heads=4, mlp_dim=dim_embeddings * 2, num_tactiles=2)
        self.mlp = nn.Sequential(
            nn.Linear(dim_embeddings * 2, dim_embeddings * 2), nn.ReLU(), nn.Dropout(0.1),
            nn.Linear(dim_embeddings * 2, dim_embeddings * 2), nn.ReLU(), nn.Dropout(0.1),
            nn.Linear(dim_embeddings * 2, dim_embeddings))
        self.query = nn.Parameter(torch.randn(1, 1, dim_embeddings))
        self.query_projection = nn.Linear(dim_embeddings, dim_embeddings)
        self.key_projection = nn.Linear(dim_embeddings, dim_embeddings)

    def forward(self, observations):
        dev = self.mae_model.mask_token.device
        obs = {k: torch.as_tensor(v).to(dev) for k, v in observations.items() if k in ('image', 'tactile')}
        latents = super().forward(dict(obs))                                     # (B, dim): MAE chain on the kernel path
        views = vt_load_lazy({'image': obs['image']}, frame_stack=self.frame_stack)
        cls = self.dino_model(mid_frame_view(views['image'], self.frame_stack))  # (B, dim): frozen, no grad
        return self.mlp(torch.cat((latents, cls.to(latents.dtype)), dim=-1))
