"""Drop-in `VTT` / `VTMAE` / `EarlyCNN` / `Transformer` modules with the reference's constructor
arguments, attribute names, obs-dict inputs, loss / latent outputs and state_dict layout
(/root/reference/models/pretrain_models.py:37-56,59-143,717-786; vit_pytorch.vit.Transformer),
computing through the sm_100a kernels behind the C-ABI.  There is no CPU path: calling a module
whose parameters are not on a CUDA device raises.

    from m3l_b200 import VTT, VTMAE        # instead of: from models.pretrain_models import VTT, VTMAE

Extra (optional) argument for parity testing: `forward(x, ..., noise=...)` supplies the uniform
draws the reference takes from torch.rand (image, tactile1, tactile2 order; pretrain_models.py:229,237).
"""
from __future__ import annotations

import math
import weakref
import random
from types import SimpleNamespace
from typing import Dict, Optional

import numpy as np
import torch
from torch import nn

from . import engine, ops
from ._lib import M3LError
from .arena import ParamArena
from .data import RawMap, clone_inputs, copy_inputs, input_signature, vt_load_lazy


def pair(t):
    return t if isinstance(t, tuple) else (t, t)


# --------------------------------------------------------------------------------------------
# parameter containers mirroring vit_pytorch's module tree (names matter for state_dict parity)
# --------------------------------------------------------------------------------------------
class FeedForward(nn.Module):
    def __init__(self, dim, hidden_dim, dropout=0.0):
        super().__init__()
        self.net = nn.Sequential(nn.LayerNorm(dim), nn.Linear(dim, hidden_dim), nn.GELU(), nn.Dropout(dropout),
                                 nn.Linear(hidden_dim, dim), nn.Dropout(dropout))


class Attention(nn.Module):
    def __init__(self, dim, heads=8, dim_head=64, dropout=0.0):
        super().__init__()
        inner = dim_head * heads
        self.heads, self.dim_head = heads, dim_head
        self.scale = dim_head ** -0.5
        self.norm = nn.LayerNorm(dim)
        self.attend = nn.Softmax(dim=-1)
        self.dropout = nn.Dropout(dropout)
        self.to_qkv = nn.Linear(dim, inner * 3, bias=False)
        if heads == 1 and dim_head == dim:
            raise M3LError("heads == 1 with dim_head == dim (identity output projection) is not supported")
        self.to_out = nn.Sequential(nn.Linear(inner, dim), nn.Dropout(dropout))


class Transformer(nn.Module):
    """vit_pytorch.vit.Transformer(dim, depth, heads, dim_head, mlp_dim, dropout=0.)."""

    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout=0.0):
        super().__init__()
        if dim_head not in ops.ATTENTION_HEAD_DIMS:
            raise M3LError(f"dim_head={dim_head}: the sm_100a attention kernels support dim_head in "
                           f"{ops.ATTENTION_HEAD_DIMS} only")
        self.dim, self.depth, self.heads, self.dim_head, self.mlp_dim, self.p_drop = dim, depth, heads, dim_head, mlp_dim, dropout
        self.norm = nn.LayerNorm(dim)
        self.layers = nn.ModuleList([])
        for _ in range(depth):
            self.layers.append(nn.ModuleList([Attention(dim, heads=heads, dim_head=dim_head, dropout=dropout),
                                              FeedForward(dim, mlp_dim, dropout=dropout)]))
        self._arena: Optional[ParamArena] = None

    def _own_arena(self) -> ParamArena:
        dev = self.norm.weight.device
        if dev.type != "cuda":
            raise M3LError("m3l_b200.Transformer needs CUDA parameters (there is no CPU fallback)")
        if self._arena is None or self._arena.device != dev:
            self._arena = ParamArena([("t." + k, p) for k, p in self.named_parameters()], dev)
        self._arena.sync()
        return self._arena

    def forward(self, x):
        """x: (B, n, dim) -> (B, n, dim); differentiable w.r.t. x and the parameters."""
        A = self._own_arena()
        spec = engine.StackSpec("t", self.dim, self.depth, self.heads, self.dim_head, self.mlp_dim)
        names = list(A.names)
        return _TransformerFn.apply(self, A, spec, x, *[A.params[n] for n in names])


class _TransformerFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mod, A, spec, x, *params):
        B, n, D = x.shape
        need = any(ctx.needs_input_grad)
        xb = x.detach().reshape(B * n, D).to(torch.bfloat16).contiguous()
        saved = [] if need else None
        xe = engine.stack_fwd(A, spec, xb, B, n, saved, p_drop=engine.p_drop(mod))
        out, st = ops.layernorm_fwd(xe, A.f32("t.norm.weight"), A.f32("t.norm.bias"), want_stats=need)
        ctx.c = (A, spec, saved, xe, st, B, n, D)
        return out.float().reshape(B, n, D)

    @staticmethod
    def backward(ctx, gout):
        A, spec, saved, xe, st, B, n, D = ctx.c
        gflat = A.new_grad_buffer()
        G = engine.GradView(A, gflat)
        dout = gout.reshape(B * n, D).to(torch.bfloat16).contiguous()
        dxe = ops.layernorm_bwd(dout, xe, st, A.f32("t.norm.weight"), dgamma=G("t.norm.weight"), dbeta=G("t.norm.bias"),
                                dx_colsum=engine.stack_dx_colsum(G, spec, saved))
        dx = engine.stack_bwd(A, G, spec, dxe, B, n, saved)
        return (None, None, None, dx.float().reshape(B, n, D), *[A.view(gflat, nm) for nm in A.names])


class Patchify(nn.Module):
    """einops Rearrange('b c (h p1) (w p2) -> b (h w) (p1 p2 c)') (pretrain_models.py:768,775).
    Parameter-free; on the hot path the rearrangement is fused into the gather kernels."""

    def __init__(self, p1, p2):
        super().__init__()
        self.p1, self.p2 = p1, p2

    def forward(self, x):
        b, c, H, W = x.shape
        h, w = H // self.p1, W // self.p2
        return x.reshape(b, c, h, self.p1, w, self.p2).permute(0, 2, 4, 3, 5, 1).reshape(b, h * w, self.p1 * self.p2 * c)


class EarlyCNN(nn.Module):
    """Conv stem used when early_conv_masking=True (pretrain_models.py:37-56)."""

    def __init__(self, in_channels, encoder_dim, key="image"):
        super().__init__()
        self.key = key
        self.conv1 = nn.Conv2d(in_channels, encoder_dim // 8, 4, stride=2, padding=1)
        self.conv2 = nn.Conv2d(encoder_dim // 8, encoder_dim // 4, 4, stride=2, padding=1)
        if key == "image":
            self.conv3 = nn.Conv2d(encoder_dim // 4, encoder_dim // 2, 4, stride=2, padding=1)
        else:
            self.conv3 = nn.Conv2d(encoder_dim // 4, encoder_dim // 2, 3, stride=1, padding=1)
        self.conv4 = nn.Conv2d(encoder_dim // 2, encoder_dim, 1)


class VTT(nn.Module):
    """Encoder container (pretrain_models.py:717-786): patch embeddings, learned positions and the
    transformer.  Same keyword-only constructor as the reference."""

    def __init__(self, *, image_size, tactile_size, image_patch_size, tactile_patch_size, dim, depth, heads, mlp_dim,
                 image_channels=3, tactile_channels=3, dim_head=64, dropout=0., emb_dropout=0, num_tactiles=2,
                 frame_stack=1):
        super().__init__()
        image_height, image_width = pair(image_size)
        tactile_height, tactile_width = pair(tactile_size)
        image_patch_height, image_patch_width = pair(image_patch_size)
        tactile_patch_height, tactile_patch_width = pair(tactile_patch_size)
        self.image_height, self.image_width = image_height, image_width
        self.tactile_height, self.tactile_width = tactile_height, tactile_width
        self.image_patch_height, self.image_patch_width = image_patch_height, image_patch_width
        self.tactile_patch_height, self.tactile_patch_width = tactile_patch_height, tactile_patch_width
        self.image_channels, self.tactile_channels = image_channels, tactile_channels
        self.frame_stack = frame_stack
        assert image_height % image_patch_height == 0 and image_width % image_patch_width == 0, \
            'Image dimensions must be divisible by the patch size.'
        assert tactile_height % tactile_patch_height == 0 and tactile_width % tactile_patch_width == 0, \
            'Tactile dimensions must be divisible by the patch size.'
        num_patches_image = (image_height // image_patch_height) * (image_width // image_patch_width)
        num_patches_tactile = (tactile_height // tactile_patch_height) * (tactile_width // tactile_patch_width) * num_tactiles
        num_patches = num_patches_image + num_patches_tactile
        image_patch_dim = image_channels * image_patch_height * image_patch_width
        tactile_patch_dim = tactile_channels * tactile_patch_height * tactile_patch_width
        self.image_to_patch_embedding = nn.Sequential(
            Patchify(image_patch_height, image_patch_width), nn.LayerNorm(image_patch_dim),
            nn.Linear(image_patch_dim, dim), nn.LayerNorm(dim))
        self.tactile_to_patch_embedding = nn.Sequential(
            Patchify(tactile_patch_height, tactile_patch_width), nn.LayerNorm(tactile_patch_dim),
            nn.Linear(tactile_patch_dim, dim), nn.LayerNorm(dim))
        self.pos_embedding = nn.Parameter(torch.randn(1, num_patches + 1, dim))
        self.dropout = nn.Dropout(emb_dropout)
        self.transformer = Transformer(dim, depth, heads, dim_head, mlp_dim, dropout)
        self.to_latent = nn.Identity()


def _as_map(t):
    """fp32 NCHW tensor of a model input (materialises a raw-observation view: m3l_vt_load kernel)."""
    return t.materialize() if isinstance(t, RawMap) else t


def _sincos_2d(nx: int, ny: int, gen_channels: int, out_channels: int) -> torch.Tensor:
    """Fixed 2-D sin/cos table as positional_encodings.PositionalEncoding2D(gen_channels) produces for a
    (1, nx, ny, out_channels) input, flattened to (nx*ny, C) (pretrain_models.py:120-140): interleaved
    sin/cos of pos * 10000^(-2i/ch); first ch channels encode the row, next ch the column."""
    ch = int(math.ceil(gen_channels / 4) * 2)
    inv_freq = 1.0 / (10000 ** (torch.arange(0, ch, 2).float() / ch))

    def enc(n):
        ang = torch.arange(n, dtype=torch.float32)[:, None] * inv_freq[None, :]
        return torch.stack((ang.sin(), ang.cos()), dim=-1).flatten(-2, -1)

    emb = torch.zeros(nx, ny, 2 * ch)
    emb[:, :, :ch] = enc(nx)[:, None, :]
    emb[:, :, ch:] = enc(ny)[None, :, :]
    return emb[:, :, :out_channels].reshape(nx * ny, -1)


class VTMAE(nn.Module):
    """Masked multimodal autoencoder (pretrain_models.py:59-715), same keyword-only constructor."""

    def __init__(self, *, encoder, decoder_dim, masking_ratio=0.75, decoder_depth=1, decoder_heads=8,
                 decoder_dim_head=64, num_tactiles=2, early_conv_masking=False, use_sincosmod_encodings=True,
                 frame_stack=1):
        super().__init__()
        assert masking_ratio > 0 and masking_ratio < 1, 'masking ratio must be kept between 0 and 1'
        self.masking_ratio = masking_ratio
        self.num_tactiles = num_tactiles
        self.frame_stack = frame_stack
        self.encoder = encoder
        num_patches, encoder_dim = encoder.pos_embedding.shape[-2:]
        num_decoder_patches = num_patches - 1
        self.use_sincosmod_encodings = use_sincosmod_encodings
        self.early_conv_masking = early_conv_masking
        if self.early_conv_masking:
            self.early_conv_vision = EarlyCNN(self.encoder.image_channels, encoder_dim, key='image')
            self.early_conv_tactile = EarlyCNN(self.encoder.tactile_channels, encoder_dim, key='tactile')
        self.image_to_patch = encoder.image_to_patch_embedding[0]
        self.image_patch_to_emb = nn.Sequential(*encoder.image_to_patch_embedding[1:])
        pixel_values_per_patch = encoder.image_to_patch_embedding[2].weight.shape[-1]
        self.tactile_to_patch = encoder.tactile_to_patch_embedding[0]
        self.tactile_patch_to_emb = nn.Sequential(*encoder.tactile_to_patch_embedding[1:])
        tactile_values_per_patch = encoder.tactile_to_patch_embedding[2].weight.shape[-1]
        self.encoder_dim = encoder_dim
        self.decoder_dim = decoder_dim
        self.enc_to_dec = nn.Linear(encoder_dim, decoder_dim) if encoder_dim != decoder_dim else nn.Identity()
        self.mask_token = nn.Parameter(torch.randn(decoder_dim))
        self.decoder = Transformer(dim=decoder_dim, depth=decoder_depth, heads=decoder_heads,
                                   dim_head=decoder_dim_head, mlp_dim=decoder_dim * 4)
        self.decoder_pos_emb = nn.Embedding(num_decoder_patches, decoder_dim)
        self.to_pixels = nn.Linear(decoder_dim, pixel_values_per_patch)
        self.to_tactiles = nn.Linear(decoder_dim, tactile_values_per_patch)
        e = self.encoder
        gi = (e.image_height // e.image_patch_height, e.image_width // e.image_patch_width)
        gt = (e.tactile_height // e.tactile_patch_height, e.tactile_width // e.tactile_patch_width)
        self.register_buffer('image_enc_pos_embedding', _sincos_2d(*gi, encoder_dim, encoder_dim)[None])
        self.register_buffer('tactile_enc_pos_embedding',
                             _sincos_2d(*gt, encoder_dim, encoder_dim).repeat(num_tactiles, 1)[None])
        self.register_buffer('image_dec_pos_embedding', _sincos_2d(*gi, encoder_dim, decoder_dim)[None])
        self.register_buffer('tactile_dec_pos_embedding',
                             _sincos_2d(*gt, encoder_dim, decoder_dim).repeat(num_tactiles, 1)[None])
        self.encoder_modality_embedding = nn.Embedding((1 + self.num_tactiles), encoder_dim)
        self.decoder_modality_embedding = nn.Embedding((1 + self.num_tactiles), decoder_dim)

        # ---- derived constants for the kernel path
        self.cfg = SimpleNamespace(
            dim=encoder_dim, decoder_dim=decoder_dim, masking_ratio=masking_ratio, num_tactiles=num_tactiles,
            n_img=gi[0] * gi[1], n_tac=gt[0] * gt[1], use_sincosmod_encodings=use_sincosmod_encodings,
            early_conv_masking=early_conv_masking, p_img=pixel_values_per_patch, p_tac=tactile_values_per_patch)
        self.ph_img, self.pw_img = e.image_patch_height, e.image_patch_width
        self.ph_tac, self.pw_tac = e.tactile_patch_height, e.tactile_patch_width
        t = e.transformer
        self.enc_spec = engine.StackSpec("encoder.transformer", t.dim, t.depth, t.heads, t.dim_head, t.mlp_dim)
        d = self.decoder
        self.dec_spec = engine.StackSpec("decoder", d.dim, d.depth, d.heads, d.dim_head, d.mlp_dim)
        self.has_enc_to_dec = encoder_dim != decoder_dim
        self.arena: Optional[ParamArena] = None
        self._tables: Dict = {}
        self._trainer = None
        self.use_cuda_graph = True      # replay mae(x) / .backward() from CUDA graphs (see _MAEGraphFn)
        self.last_masked_indices = self.last_unmasked_indices = None

    # ------------------------------------------------------------------------------ plumbing
    def _canonical_named_params(self):
        """(name, param) in arena order: decoder-side first (their gradients are final first in the
        backward pass), then encoder side; shared patch-embedding modules once, under the
        `*_patch_to_emb` names."""
        named = dict(self.named_parameters(remove_duplicate=False))
        dec_side = [k for k in named if k.startswith(("to_pixels", "to_tactiles", "decoder.", "mask_token",
                                                      "decoder_modality_embedding", "enc_to_dec"))]
        skip = ("encoder.image_to_patch_embedding", "encoder.tactile_to_patch_embedding")
        rest = [k for k in named if k not in dec_side and not k.startswith(skip)]
        return [(k, named[k]) for k in dec_side + rest]

    LATE = ("encoder.pos_embedding", "decoder_pos_emb.weight")

    def _sync(self) -> ParamArena:
        dev = self.mask_token.device
        if dev.type != "cuda":
            raise M3LError("m3l_b200.VTMAE needs its parameters on a CUDA device: the compute path is the sm_100a "
                           "kernel library and there is no CPU fallback (call .cuda() first)")
        if self.arena is None or self.arena.device != dev:
            dead = ("image_patch_to_emb", "tactile_patch_to_emb") if self.early_conv_masking else ("early_conv",)
            late = [k for k, _ in self._canonical_named_params()
                    if (k in self.LATE and self.use_sincosmod_encodings) or k.startswith(dead)]
            self.arena = ParamArena(self._canonical_named_params(), dev, late_names=late)
            self._tables = {}
            self._trainer = None
            self.__dict__.pop("_mae_graphs", None)      # captured graphs point into the old arena
        self.arena.sync()
        return self.arena

    def tables(self, geo, B):
        key = (geo.use_vision, geo.nt, B)
        if key not in self._tables:
            self._tables[key] = engine.Tables(self, geo, B, self.arena.device)
        return self._tables[key]

    def live_param_names(self, geo, masked: bool):
        """Parameters that receive a gradient in this mode (the reference leaves .grad None on the rest)."""
        names = []
        for k in self.arena.names:
            if k.startswith("early_conv_vision") and not (self.early_conv_masking and geo.use_vision):
                continue
            if k.startswith("early_conv_tactile") and not (self.early_conv_masking and geo.nt):
                continue
            if k.startswith(("image_patch_to_emb", "tactile_patch_to_emb")) and self.early_conv_masking:
                continue  # the conv stems replace the patch embeddings (pretrain_models.py:180-191)
            if k == "encoder.pos_embedding" and self.use_sincosmod_encodings:
                continue
            if k == "decoder_pos_emb.weight" and (self.use_sincosmod_encodings or not masked):
                continue
            if k == "encoder_modality_embedding.weight" and not self.use_sincosmod_encodings:
                continue
            if k == "decoder_modality_embedding.weight" and (not self.use_sincosmod_encodings or not masked):
                continue
            if k.startswith("image_patch_to_emb") and not geo.use_vision:
                continue
            if k.startswith("tactile_patch_to_emb") and not geo.nt:
                continue
            if k.startswith("to_pixels") and not (geo.use_vision and masked):
                continue
            if k.startswith("to_tactiles") and not (geo.nt and masked):
                continue
            if not masked and k.startswith(("decoder.", "mask_token", "enc_to_dec")):
                continue
            names.append(k)
        return names

    def _prep_inputs(self, x, use_vision, use_tactile, reconstruct_ratio=None):
        if 'image' not in x:
            use_vision = False
        geo = engine.make_geometry(self.cfg, use_vision, use_tactile, reconstruct_ratio)
        xs = {}
        keys = (['image'] if geo.use_vision else []) + [f'tactile{i + 1}' for i in range(geo.nt)]
        for k in keys:
            t = x[k]
            if not t.is_cuda:
                raise M3LError(f"input '{k}' is not on a CUDA device (no CPU fallback)")
            # data.RawMap: a view into the raw observation tensor; vt_load happens inside the patch-gather kernels
            xs[k] = t if isinstance(t, RawMap) else t.detach().to(torch.float32).contiguous()
        B = xs[keys[0]].shape[0]
        return xs, geo, B

    # ------------------------------------------------------------------------------ reference API
    def forward(self, x, use_vision=True, use_tactile=True, noise=None):
        """Masked reconstruction loss (0-dim fp32 tensor with grad_fn), pretrain_models.py:146-342."""
        A = self._sync()
        xs, geo, B = self._prep_inputs(x, use_vision, use_tactile)
        if noise is None:
            noise = torch.rand(B, geo.n, device=A.device)
        noise = noise.to(device=A.device, dtype=torch.float32).contiguous()
        assert noise.shape == (B, geo.n), f"noise must be ({B}, {geo.n})"
        live = self.live_param_names(geo, True)
        params = [A.params[k] for k in live]
        if self.use_cuda_graph and torch.is_grad_enabled() and any(p.requires_grad for p in params):
            key = ("mae", geo.use_vision, geo.nt, B, input_signature(xs), engine.p_drop(self.encoder.transformer))
            # The graph entry owns ONE set of saved activations.  If the previous replayed forward of this shape has
            # not been back-propagated yet (two forwards before a backward: SAC with a shared extractor, gradient
            # accumulation over two losses), this call takes the eager autograd path, which owns its activations.
            if _entry_free(self.__dict__.get("_mae_graphs", {}).get(key)):
                ent = _graph_entry(self, key, xs, noise, geo)
                return _MAEGraphFn.apply(self, ent, geo, tuple(live), *params)
        return _MAEFn.apply(self, xs, noise, geo, tuple(live), *params)

    def get_embeddings(self, x, eval=True, use_vision=True, use_tactile=True):
        """Encoder over all tokens, no masking (pretrain_models.py:588-668) -> (B, N, dim) fp32."""
        if eval:
            self.eval()
        else:
            self.train()
        A = self._sync()
        xs, geo, B = self._prep_inputs(x, use_vision, use_tactile)
        live = self.live_param_names(geo, False)
        params = [A.params[k] for k in live]
        if self.use_cuda_graph and torch.is_grad_enabled() and any(p.requires_grad for p in params):
            cache = self.__dict__.setdefault("_mae_graphs", {})
            key = ("emb", geo.use_vision, geo.nt, B, input_signature(xs), engine.p_drop(self.encoder.transformer))
            ent = cache.get(key)
            if _entry_free(ent):                  # else: previous forward not back-propagated yet -> eager path
                if ent is None:
                    if len(cache) >= _MAX_GRAPHS:
                        cache.pop(next(iter(cache)))
                    ent = cache[key] = _capture_emb_graphs(self, xs, geo, B)
                copy_inputs(ent.xs, xs)
                return _EmbGraphFn.apply(self, ent, tuple(live), *params)
        return _EmbFn.apply(self, xs, geo, B, tuple(live), *params)

    @torch.no_grad()
    def reconstruct(self, x, mask_ratio=None, use_vision=True, use_tactile=True, noise=None):
        """Visualisation helper (pretrain_models.py:344-586): masks `int(mask_ratio * 64)` patches PER MODALITY
        (a different split rule from forward()), runs encoder + decoder + heads through the kernels and
        returns the reference's dict: image_rec / image_masked (masked patches = 0.5) / recon_loss_image,
        tactile_rec / tactile_masked (masked patches = inf) / recon_loss_tactile.  The patch <-> map
        rearrangements of the outputs are torch indexing ops (not on the hot path); values are detached."""
        if mask_ratio is None:
            mask_ratio = self.masking_ratio
        A = self._sync()
        xs, geo, B = self._prep_inputs(x, use_vision, use_tactile, reconstruct_ratio=mask_ratio)
        if noise is None:
            noise = torch.rand(B, geo.n, device=A.device)
        noise = noise.to(device=A.device, dtype=torch.float32).contiguous()
        assert noise.shape == (B, geo.n), f"noise must be ({B}, {geo.n})"
        cap = {}
        engine.mae_forward(self, xs, noise, geo, training=False, capture=cap)
        masked = self.last_masked_indices
        br = torch.arange(B, device=A.device)[:, None]
        e = self.encoder
        out = {}
        if geo.use_vision:
            gh, gw = e.image_height // self.ph_img, e.image_width // self.pw_img
            patches = self.image_to_patch(_as_map(xs['image']))
            mi = masked[:, :geo.nm_img]
            vis, rec = patches.clone(), patches.clone()
            vis[br, mi] = 0.5
            if self.early_conv_masking:      # heads on ALL tokens; the reconstruction is the prediction (:560-567)
                rec = cap["pred_image"].view(B, geo.n_img, -1)
                out['recon_loss_image'] = torch.nn.functional.mse_loss(rec, patches)
            else:
                pred = cap["pred_image"].view(B, geo.nm_img, -1)
                out['recon_loss_image'] = torch.nn.functional.mse_loss(pred, patches[br, mi])
                rec[br, mi] = pred
            unp = lambda t: t.reshape(B, gh, gw, self.ph_img, self.pw_img, -1).permute(0, 5, 1, 3, 2, 4).reshape(
                B, -1, gh * self.ph_img, gw * self.pw_img)       # 'b (h w) (p1 p2 c) -> b c (h p1) (w p2)'
            out['image_rec'], out['image_masked'] = unp(rec), unp(vis)
        if geo.nt:
            gh, gw = e.tactile_height // self.ph_tac, e.tactile_width // self.pw_tac
            patches = torch.cat([self.tactile_to_patch(_as_map(xs[f'tactile{i + 1}'])) for i in range(geo.nt)], dim=1)
            mt = masked[:, geo.nm_img:] - geo.n_img
            vis, rec = patches.clone(), patches.clone()
            vis[br, mt] = float('inf')
            if self.early_conv_masking:
                rec = cap["pred_tactile"].view(B, geo.nt * geo.n_tac, -1)
                out['recon_loss_tactile'] = torch.nn.functional.mse_loss(rec, patches)
            else:
                pred = cap["pred_tactile"].view(B, geo.nm_tac_total, -1)
                out['recon_loss_tactile'] = torch.nn.functional.mse_loss(pred, patches[br, mt])
                rec[br, mt] = pred
            unp = lambda t: t.reshape(B, geo.nt, gh, gw, self.ph_tac, self.pw_tac, -1).permute(0, 1, 6, 2, 4, 3, 5).reshape(
                B, -1, gh * self.ph_tac, gw * self.pw_tac)       # 'b (n h w) (p1 p2 c) -> b (n c) (h p1) (w p2)'
            out['tactile_rec'], out['tactile_masked'] = unp(rec), unp(vis)
        order = ['image_rec', 'image_masked', 'recon_loss_image', 'tactile_rec', 'tactile_masked', 'recon_loss_tactile']
        return {k: out[k] for k in order if k in out}

    def initialize_training(self, train_args):
        """pretrain_models.py:670-676: AdamW(lr) + batch size; the optimizer is the fused flat-arena one."""
        from .trainer import FusedTrainer
        self._sync()
        self.batch_size = train_args['batch_size']
        self._trainer = FusedTrainer(self, lr=train_args['lr'])
        self.optimizer = self._trainer.optimizer_facade()

    def train_step(self, x, noise=None, use_vision=True, use_tactile=True):
        """zero_grad + forward + backward + clip_grad_norm_(0.5) + AdamW.step (pretrain_models.py:707-711)
        as one fused kernel sequence.  Returns the loss (device tensor, no sync)."""
        if self._trainer is None:
            raise M3LError("call initialize_training({'lr': ..., 'batch_size': ...}) first")
        return self._trainer.step(x, noise=noise, use_vision=use_vision, use_tactile=use_tactile)

    def train_iterations(self, iterations, replay_buffer, no_tactile=False):
        """pretrain_models.py:679-715 (host-side batch assembly kept as in the reference)."""
        if len(replay_buffer) < self.batch_size:
            print("Not enough samples in replay buffer")
            return
        self.train()
        for _ in range(iterations):
            xb = random.choices(replay_buffer, k=self.batch_size)
            new_x = {}
            keys = ['image'] if no_tactile else ['image', 'tactile']
            for key in keys:
                new_x[key] = np.stack([xb[j][key] for j in range(self.batch_size)])
            if 'image' in new_x:
                new_x['image'] = new_x['image'].transpose((0, 2, 3, 1, 4))
                new_x['image'] = new_x['image'].reshape((new_x['image'].shape[0], new_x['image'].shape[1], new_x['image'].shape[2], -1))
            if 'tactile' in new_x:
                new_x['tactile'] = new_x['tactile'].reshape((new_x['tactile'].shape[0], -1, new_x['tactile'].shape[3], new_x['tactile'].shape[4]))
            # raw batch -> device; vt_load itself (layout, de-interleave, normalisation) runs inside the patch gathers
            xd = vt_load_lazy(new_x, frame_stack=self.frame_stack, device=self.mask_token.device)
            self.train_step(xd)
        self.eval()


# --------------------------------------------------------------------------------------------
# rollout feature extractor (pretrain_models.py:788-841)
# --------------------------------------------------------------------------------------------
try:                                       # SB3 only reads `.features_dim`; it is optional here
    from stable_baselines3.common.torch_layers import BaseFeaturesExtractor as _ExtractorBase
except Exception:                          # pragma: no cover - SB3 is not part of this image
    class _ExtractorBase(nn.Module):
        def __init__(self, observation_space, features_dim: int = 0):
            super().__init__()
            assert features_dim > 0
            self._observation_space = observation_space
            self._features_dim = features_dim

        @property
        def features_dim(self) -> int:
            return self._features_dim


class MAEExtractor(_ExtractorBase):
    """SB3 features extractor of the PPO / SAC policies: obs dict -> MAE encoder over all tokens (no
    masking) -> one extra transformer block (`vit_layer.transformer`) -> mean over tokens -> (B, dim).
    Same constructor and attributes as the reference (pretrain_models.py:788-841); `vit_layer` is a
    full VTT of which only `.transformer` is used (its other parameters exist in the state_dict and
    never receive gradients, as in the reference).  The whole chain runs as one kernel sequence
    (bf16 hand-off between the encoder, the extra block and the token mean) and is differentiable
    w.r.t. the MAE and the extra block, as the PPO / SAC losses need (ppo_mae.py:280,340)."""

    def __init__(self, observation_space, mae_model, dim_embeddings, vision_only_control, frame_stack) -> None:
        super().__init__(observation_space, dim_embeddings)
        self.flatten = nn.Flatten()
        self.mae_model = mae_model
        self.running_buffer = {}
        self.vision_only_control = vision_only_control
        self.frame_stack = frame_stack
        self.vit_layer = VTT(image_size=(64, 64), tactile_size=(32, 32), image_patch_size=8, tactile_patch_size=4,
                             dim=dim_embeddings, depth=1, heads=4, mlp_dim=dim_embeddings * 2, num_tactiles=2)

    def forward(self, observations):
        mae = self.mae_model
        dev = mae.mask_token.device
        obs = {k: torch.as_tensor(v).to(dev) for k, v in observations.items() if k in ('image', 'tactile')}
        cached = self.__dict__.get("_joint_feats")
        if cached is not None:                                    # features of joint_mae_loss() on these very observations
            self._joint_feats = None
            if cached[0] == _obs_key(obs) and torch.is_grad_enabled():
                return self.flatten(cached[1])
        if getattr(self, "use_cuda_graph", True):
            if not torch.is_grad_enabled():
                return self._forward_graph(obs)
            if any(p.requires_grad for p in self.parameters()):
                return self._forward_graph_grad(obs)
        return self._forward_eager(obs)

    def joint_mae_loss(self, observations, noise=None):
        """The two passes a PPO / SAC minibatch makes over the SAME observations (ppo_mae.py:255-283: `mae(x)` with
        backward, then `evaluate_actions` -> this extractor with backward) as ONE pass: the patch embedding of all tokens
        is computed once, the masked encoder reads its visible rows from it, and in the backward pass the two gradients
        meet before a single embedding backward.  Returns the MAE loss; the extractor features of the same pass are
        handed out by the next `forward(observations)` on these observations (the call `evaluate_actions` makes), both
        attached to one autograd node, so `(ppo_loss + mae_loss).backward()` replays one backward graph.
        Falls back to `mae(vt_load(obs))` when the extractor uses a different token set (vision_only_control)."""
        mae = self.mae_model
        dev = mae.mask_token.device
        obs = {k: torch.as_tensor(v).to(dev) for k, v in observations.items() if k in ('image', 'tactile')}
        if self.vision_only_control or not torch.is_grad_enabled():
            return mae(vt_load_lazy(obs, frame_stack=self.frame_stack), noise=noise)
        mae.train()
        A = mae._sync()
        Av = self.vit_layer.transformer._own_arena()
        xs, geo, B, _, _ = self._prep(dict(obs))
        if noise is None:
            noise = torch.rand(B, geo.n, device=dev)
        noise = noise.to(device=dev, dtype=torch.float32).contiguous()
        key = ("joint",) + tuple((k, tuple(v.shape), v.dtype) for k, v in sorted(obs.items())) + (id(A), id(Av)) + \
              self._p_drops()
        cache = self.__dict__.setdefault("_graphs", {})
        ent = cache.get(key)
        if not _entry_free(ent):
            ent_fn, args = _JointFn, (self, xs, noise, geo, B)
        else:
            if ent is None:
                if len(cache) >= 8:
                    cache.pop(next(iter(cache)))
                ent = cache[key] = _capture_joint_graphs(self, obs, noise)
            for k, v in obs.items():
                ent.xs[k].copy_(v, non_blocking=True)
            ent.noise.copy_(noise, non_blocking=True)
            ent_fn, args = _JointGraphFn, (self, ent)
        live = tuple(mae.live_param_names(geo, True))
        vit_names = tuple(Av.names)
        loss, feats = ent_fn.apply(*args, live, vit_names, *[A.params[k] for k in live], *[Av.params[k] for k in vit_names])
        self._joint_feats = (_obs_key(obs), feats)
        return loss

    def _forward_graph_grad(self, obs):
        """Training-time call (PPO / SAC evaluate the policy on a minibatch and back-propagate through the extractor:
        ppo_mae.py:280,340): forward and backward replayed from two CUDA graphs sharing one memory pool."""
        mae = self.mae_model
        mae.train()                                               # get_embeddings(eval=False) side effect (:590-593)
        A = mae._sync()
        Av = self.vit_layer.transformer._own_arena()
        key = ("grad",) + tuple((k, tuple(v.shape), v.dtype) for k, v in sorted(obs.items())) + \
              (bool(self.vision_only_control), id(A), id(Av)) + self._p_drops()
        cache = self.__dict__.setdefault("_graphs", {})
        ent = cache.get(key)
        if not _entry_free(ent):                  # previous forward of this shape not back-propagated yet
            return self._forward_eager(obs)
        if ent is None:
            if len(cache) >= 8:
                cache.pop(next(iter(cache)))
            ent = cache[key] = _capture_extractor_graphs(self, obs)
        for k, v in obs.items():
            ent.xs[k].copy_(v, non_blocking=True)
        return self.flatten(_ExtractorGraphFn.apply(self, ent, ent.live, ent.vit_names,
                                                    *[A.params[k] for k in ent.live], *[Av.params[k] for k in ent.vit_names]))

    def _forward_graph(self, obs):
        """Rollout-time inference (torch.no_grad): the whole chain — observation reshapes, vt_load, encoder, extra
        block, token mean — replayed from a CUDA graph cached per observation shape.  A rollout step with a handful of
        environments is launch-bound (≈ 60 kernels): 1.95 ms eager -> see tools/rollout_latency.py."""
        mae = self.mae_model
        key = tuple((k, tuple(v.shape), v.dtype) for k, v in sorted(obs.items())) + (bool(self.vision_only_control),)
        cache = self.__dict__.setdefault("_graphs", {})
        ent = cache.get(key)
        mae.train()                                               # get_embeddings(eval=False) side effect (:590-593)
        A = mae._sync()                                           # bf16 shadows current (outside the graph)
        Av = self.vit_layer.transformer._own_arena()
        key = key + (id(A), id(Av))                               # a re-created arena invalidates captured pointers
        key = key + self._p_drops()                               # the dropout of a graph is fixed at capture
        ent = cache.get(key)
        if ent is None:
            static_in = {k: v.clone() for k, v in obs.items()}
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):                            # warm-up: lazy tables / kernel attributes / allocator
                self._forward_eager(dict(static_in))
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with engine.capture_guard(), torch.cuda.graph(g):
                out = self._forward_eager(dict(static_in))
            ent = cache[key] = (g, static_in, out)
        g, static_in, out = ent
        for k, v in obs.items():
            static_in[k].copy_(v, non_blocking=True)
        g.replay()
        return out.clone()

    def _forward_eager(self, obs):
        xs, geo, B, A, Av = self._prep(obs)
        live = self.mae_model.live_param_names(geo, False)
        vit_names = list(Av.names)
        out = _ExtractorFn.apply(self, xs, geo, B, tuple(live), tuple(vit_names),
                                 *[A.params[k] for k in live], *[Av.params[k] for k in vit_names])
        return self.flatten(out)

    def _prep(self, obs):
        """Observation reshapes (pretrain_models.py:823-827) + vt_load -> (model inputs, geometry, batch, arenas)."""
        mae = self.mae_model
        # The 5-D frame-stack reshapes (:823-827) and vt_load are not executed: the observation tensors stay as the
        # rollout buffer holds them and the patch-gather kernels read them in place (data.RawMap, layout 1).
        if mae.early_conv_masking:
            vt = {k: v.materialize() for k, v in vt_load_lazy(obs, frame_stack=self.frame_stack).items()}
        else:
            vt = vt_load_lazy(obs, frame_stack=self.frame_stack)
        mae.train()                                               # get_embeddings(eval=False) side effect (:590-593)
        A = mae._sync()
        xs, geo, B = mae._prep_inputs(vt, True, not self.vision_only_control)
        Av = self.vit_layer.transformer._own_arena()
        return xs, geo, B, A, Av

    def _p_drops(self):
        """Dropout probabilities in force for the MAE encoder and the extra block (part of every graph key).  The MAE
        runs in training mode here (get_embeddings(eval=False) in the reference), so its encoder dropout applies."""
        return engine.p_drop(self.mae_model.encoder.transformer), engine.p_drop(self.vit_layer.transformer)


class _ExtractorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ext, xs, geo, B, live, vit_names, *params):
        mae, tr = ext.mae_model, ext.vit_layer.transformer
        Av = tr._arena
        need = any(ctx.needs_input_grad)
        emb, c = engine.embeddings_forward(mae, xs, geo, B, training=need)
        spec = engine.StackSpec("t", tr.dim, tr.depth, tr.heads, tr.dim_head, tr.mlp_dim)
        saved = [] if need else None
        xe = engine.stack_fwd(Av, spec, emb, B, geo.n, saved, p_drop=engine.p_drop(tr))
        y, st = ops.layernorm_fwd(xe, Av.f32("t.norm.weight"), Av.f32("t.norm.bias"), want_stats=need)
        out = ops.token_mean_fwd(y, B, geo.n)
        ctx.c = (mae, Av, spec, c, saved, xe, st, B, geo.n, live, vit_names)
        return out

    @staticmethod
    def backward(ctx, gout):
        mae, Av, spec, c, saved, xe, st, B, n, live, vit_names = ctx.c
        A = mae.arena
        dy = ops.token_mean_bwd(gout.to(torch.float32).contiguous(), B, n)
        gv = Av.new_grad_buffer()
        Gv = engine.GradView(Av, gv)
        dxe = ops.layernorm_bwd(dy, xe, st, Av.f32("t.norm.weight"), dgamma=Gv("t.norm.weight"), dbeta=Gv("t.norm.bias"),
                                dx_colsum=engine.stack_dx_colsum(Gv, spec, saved))
        demb = engine.stack_bwd(Av, Gv, spec, dxe, B, n, saved)
        gm = A.new_grad_buffer()
        engine.embeddings_backward(mae, c, demb, gm)
        return (None, None, None, None, None, None, *[A.view(gm, k) for k in live], *[Av.view(gv, k) for k in vit_names])


def _capture_extractor_graphs(ext, obs):
    mae, tr = ext.mae_model, ext.vit_layer.transformer
    ent = _GraphEntry()
    ent.xs = {k: v.clone() for k, v in obs.items()}
    ent.gen, ent.consumed, ent.node = 0, True, None
    xs, geo, B, A, Av = ext._prep(dict(ent.xs))
    ent.live, ent.vit_names = tuple(mae.live_param_names(geo, False)), tuple(Av.names)
    ent.gflat, ent.gflat2 = A.new_grad_buffer(), Av.new_grad_buffer()
    ent.gout = torch.zeros((B, tr.dim), dtype=torch.float32, device=A.device)
    spec = engine.StackSpec("t", tr.dim, tr.depth, tr.heads, tr.dim_head, tr.mlp_dim)

    def fwd():
        xs, geo, B, _, _ = ext._prep(dict(ent.xs))
        emb, c = engine.embeddings_forward(mae, xs, geo, B, training=True)
        saved = []
        xe = engine.stack_fwd(Av, spec, emb, B, geo.n, saved, p_drop=engine.p_drop(tr))
        y, st = ops.layernorm_fwd(xe, Av.f32("t.norm.weight"), Av.f32("t.norm.bias"), want_stats=True)
        ent.loss = ops.token_mean_fwd(y, B, geo.n)
        ent.ctx = (c, saved, xe, st, B, geo.n)

    def bwd():
        c, saved, xe, st, B, n = ent.ctx
        ent.gflat.zero_()
        ent.gflat2.zero_()
        Gv = engine.GradView(Av, ent.gflat2)
        dy = ops.token_mean_bwd(ent.gout, B, n)
        dxe = ops.layernorm_bwd(dy, xe, st, Av.f32("t.norm.weight"), dgamma=Gv("t.norm.weight"), dbeta=Gv("t.norm.bias"),
                                dx_colsum=engine.stack_dx_colsum(Gv, spec, saved))
        demb = engine.stack_bwd(Av, Gv, spec, dxe, B, n, saved)
        engine.embeddings_backward(mae, c, demb, ent.gflat)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fwd()
        bwd()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    pool = torch.cuda.graph_pool_handle()
    ent.fwd, ent.bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with engine.capture_guard():
        with torch.cuda.graph(ent.fwd, pool=pool):
            fwd()
        with torch.cuda.graph(ent.bwd, pool=pool):
            bwd()
    return ent


class _ExtractorGraphFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ext, ent, live, vit_names, *params):
        ent.gen += 1
        ent.consumed = False
        ent.node = _weak(ctx)
        ent.fwd.replay()
        ctx.ext, ctx.ent, ctx.gen = ext, ent, ent.gen
        return ent.loss.clone()

    @staticmethod
    def backward(ctx, gout):
        ent = ctx.ent
        if ctx.gen != ent.gen or ent.consumed:
            raise M3LError("backward through a CUDA-graph replayed extractor forward whose saved activations were "
                           "overwritten by a newer forward of the same shape (or a second backward): set "
                           "extractor.use_cuda_graph = False for this pattern")
        ent.consumed = True
        ent.gout.copy_(gout)
        ent.bwd.replay()
        A, Av = ctx.ext.mae_model.arena, ctx.ext.vit_layer.transformer._arena
        gm, gv = ent.gflat.clone(), ent.gflat2.clone()    # .grad must never alias the graph's static buffers
        return (None, None, None, None, *[A.view(gm, k) for k in ent.live], *[Av.view(gv, k) for k in ent.vit_names])


def _obs_key(obs):
    return tuple((k, v.data_ptr(), tuple(v.shape), v.dtype, v._version) for k, v in sorted(obs.items()))


# --------------------------------------------------------------------------------------------
# joint MAE + feature-extractor pass over one minibatch (SURVEY.md section 8(f)-2; ppo_mae.py:255-283)
# --------------------------------------------------------------------------------------------
def _joint_forward(ext, xs, noise, geo, B, gflat_m):
    """-> (loss_acc [1], feats [B, dim], ctx).  gflat_m: gradient buffer of the masked-autoencoder branch."""
    mae, tr = ext.mae_model, ext.vit_layer.transformer
    Av = tr._arena
    emb, c = engine.embeddings_forward(mae, xs, geo, B, training=True)          # embeds ALL tokens once; encoder over them
    loss_acc, cm = engine.mae_forward(mae, xs, noise, geo, training=True, gflat=gflat_m, tokens_all=c["tokens_all"])
    spec = engine.StackSpec("t", tr.dim, tr.depth, tr.heads, tr.dim_head, tr.mlp_dim)
    saved = []
    xe = engine.stack_fwd(Av, spec, emb, B, geo.n, saved, p_drop=engine.p_drop(tr))
    y, st = ops.layernorm_fwd(xe, Av.f32("t.norm.weight"), Av.f32("t.norm.bias"), want_stats=True)
    feats = ops.token_mean_fwd(y, B, geo.n)
    return loss_acc, feats, (c, cm, spec, saved, xe, st, B, geo.n)


def _joint_backward(ext, ctx, g_loss, g_feats, gflat, gflat_m, gflat2):
    """gflat: MAE-arena gradients of the extractor branch and of the shared embedding; gflat_m: of the masked-autoencoder
    branch (scaled by the loss gradient, then added into gflat); gflat2: extra-block arena gradients."""
    mae, Av = ext.mae_model, ext.vit_layer.transformer._arena
    c, cm, spec, saved, xe, st, B, n = ctx
    Gv = engine.GradView(Av, gflat2)
    dy = ops.token_mean_bwd(g_feats, B, n)
    dxe = ops.layernorm_bwd(dy, xe, st, Av.f32("t.norm.weight"), dgamma=Gv("t.norm.weight"), dbeta=Gv("t.norm.bias"),
                            dx_colsum=engine.stack_dx_colsum(Gv, spec, saved))
    demb = engine.stack_bwd(Av, Gv, spec, dxe, B, n, saved)
    engine.mae_backward_decoder(mae, cm, gflat_m)
    dx0 = engine.mae_backward_encoder(mae, cm, gflat_m)
    dx0.mul_(g_loss.to(dx0.dtype))
    gflat_m.mul_(g_loss)
    engine.embeddings_backward(mae, c, demb, gflat, extra_token_grad=(dx0, cm["emb"]["unmasked32"]))
    gflat.add_(gflat_m)


class _JointFn(torch.autograd.Function):
    """Eager form (owns its activations): used when a graph-replayed joint pass is still outstanding."""

    @staticmethod
    def forward(ctx, ext, xs, noise, geo, B, live, vit_names, *params):
        A = ext.mae_model.arena
        gm = A.new_grad_buffer()
        loss_acc, feats, c = _joint_forward(ext, xs, noise, geo, B, gm)
        ctx.c = (ext, c, gm, live, vit_names)
        ext.mae_model.last_masked_indices = ext.mae_model.last_masked_indices.clone()
        return loss_acc.reshape(()), feats

    @staticmethod
    def backward(ctx, g_loss, g_feats):
        ext, c, gm, live, vit_names = ctx.c
        A, Av = ext.mae_model.arena, ext.vit_layer.transformer._arena
        g, gv = A.new_grad_buffer(), Av.new_grad_buffer()
        B, dim = c[6], ext.vit_layer.transformer.dim
        gl = g_loss if g_loss is not None else torch.zeros((), device=A.device)
        gf = g_feats.to(torch.float32).contiguous() if g_feats is not None else torch.zeros((B, dim), device=A.device)
        _joint_backward(ext, c, gl.reshape(()).to(torch.float32), gf, g, gm, gv)
        return (None,) * 7 + tuple(A.view(g, k) for k in live) + tuple(Av.view(gv, k) for k in vit_names)


def _capture_joint_graphs(ext, obs, noise):
    mae, tr = ext.mae_model, ext.vit_layer.transformer
    ent = _GraphEntry()
    ent.xs = {k: v.clone() for k, v in obs.items()}
    ent.noise = noise.clone()
    ent.gen, ent.consumed, ent.node = 0, True, None
    xs, geo, B, A, Av = ext._prep(dict(ent.xs))
    ent.live, ent.vit_names = tuple(mae.live_param_names(geo, True)), tuple(Av.names)
    ent.gflat, ent.gflat2 = A.new_grad_buffer(), Av.new_grad_buffer()
    gflat_m = A.new_grad_buffer()
    ent.gout = (torch.ones((), dtype=torch.float32, device=A.device), torch.zeros((B, tr.dim), dtype=torch.float32, device=A.device))

    def fwd():
        xs, geo, B, _, _ = ext._prep(dict(ent.xs))
        gflat_m.zero_()
        loss_acc, feats, ent.ctx = _joint_forward(ext, xs, ent.noise, geo, B, gflat_m)
        ent.loss = (loss_acc, feats)
        ent.masked, ent.unmasked = mae.last_masked_indices, mae.last_unmasked_indices

    def bwd():
        ent.gflat.zero_()
        ent.gflat2.zero_()
        _joint_backward(ext, ent.ctx, ent.gout[0], ent.gout[1], ent.gflat, gflat_m, ent.gflat2)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fwd()
        bwd()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    pool = torch.cuda.graph_pool_handle()
    ent.fwd, ent.bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with engine.capture_guard():
        with torch.cuda.graph(ent.fwd, pool=pool):
            fwd()
        with torch.cuda.graph(ent.bwd, pool=pool):
            bwd()
    return ent


class _JointGraphFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ext, ent, live, vit_names, *params):
        ent.gen += 1
        ent.consumed = False
        ent.node = _weak(ctx)
        ent.fwd.replay()
        mae = ext.mae_model
        mae.last_masked_indices, mae.last_unmasked_indices = ent.masked.clone(), ent.unmasked.clone()
        ctx.ext, ctx.ent, ctx.gen = ext, ent, ent.gen
        return ent.loss[0].reshape(()).clone(), ent.loss[1].clone()

    @staticmethod
    def backward(ctx, g_loss, g_feats):
        ent = ctx.ent
        if ctx.gen != ent.gen or ent.consumed:
            raise M3LError("backward through a CUDA-graph replayed joint pass whose saved activations were overwritten")
        ent.consumed = True
        if g_loss is not None:
            ent.gout[0].copy_(g_loss.reshape(()))
        else:
            ent.gout[0].zero_()
        if g_feats is not None:
            ent.gout[1].copy_(g_feats)
        else:
            ent.gout[1].zero_()
        ent.bwd.replay()
        A, Av = ctx.ext.mae_model.arena, ctx.ext.vit_layer.transformer._arena
        gm, gv = ent.gflat.clone(), ent.gflat2.clone()
        return (None, None, None, None, *[A.view(gm, k) for k in ent.live], *[Av.view(gv, k) for k in ent.vit_names])


# --------------------------------------------------------------------------------------------
# CUDA-graph replay of the autograd path  loss = mae(x); loss.backward()
# --------------------------------------------------------------------------------------------
# The reference's learners call the module through autograd (ppo_mae.py:262-263, sac_mae.py:284-291).  Eagerly that is
# ~165 kernel launches behind Python / ctypes calls: 6.3 ms of host time for 2.3 ms of GPU work at batch 256
# (tools/eager_latency.py).  Forward and backward are therefore captured once per (modalities, batch) as two CUDA graphs
# sharing one memory pool (the forward graph's saved activations are the backward graph's inputs) and replayed.
_MAX_GRAPHS = 4


def _weak(node):
    try:
        return weakref.ref(node)
    except TypeError:                        # not weak-referenceable: treat the forward as outstanding until consumed
        return lambda: True


def _entry_free(ent) -> bool:
    """True when a graph entry may be replayed: none captured yet, or its last forward was consumed by a backward /
    its autograd node is gone (result discarded, e.g. an evaluation-only call under enable_grad)."""
    if ent is None or ent.consumed:
        return True
    node = ent.node() if ent.node is not None else None
    return node is None


class _GraphEntry:
    __slots__ = ("fwd", "bwd", "xs", "noise", "loss", "ctx", "gflat", "gflat2", "gout", "gen", "consumed", "masked", "unmasked",
                 "live", "vit_names", "node")


def _graph_entry(model, key, xs, noise, geo):
    cache = model.__dict__.setdefault("_mae_graphs", {})
    ent = cache.get(key)
    if ent is None:
        if len(cache) >= _MAX_GRAPHS:
            cache.pop(next(iter(cache)))
        ent = cache[key] = _capture_mae_graphs(model, xs, noise, geo)
    copy_inputs(ent.xs, xs)
    ent.noise.copy_(noise, non_blocking=True)
    return ent


def _capture_mae_graphs(model, xs, noise, geo):
    A = model.arena
    ent = _GraphEntry()
    ent.xs = clone_inputs(xs)
    ent.noise = noise.clone()
    ent.gflat = A.new_grad_buffer()
    ent.gout = torch.ones((), dtype=torch.float32, device=A.device)
    ent.gen, ent.consumed, ent.node = 0, True, None

    def fwd():
        ent.gflat.zero_()
        ent.loss, ent.ctx = engine.mae_forward(model, ent.xs, ent.noise, geo, training=True, gflat=ent.gflat)
        ent.masked, ent.unmasked = model.last_masked_indices, model.last_unmasked_indices

    def bwd():
        engine.mae_backward_decoder(model, ent.ctx, ent.gflat)
        engine.mae_backward_encoder(model, ent.ctx, ent.gflat)
        ent.gflat.mul_(ent.gout)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                       # warm-up: lazy tables, kernel attributes, allocator
        fwd()
        bwd()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    pool = torch.cuda.graph_pool_handle()
    ent.fwd, ent.bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with engine.capture_guard():
        with torch.cuda.graph(ent.fwd, pool=pool):
            fwd()
        with torch.cuda.graph(ent.bwd, pool=pool):
            bwd()
    return ent


class _MAEGraphFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, ent, geo, live, *params):
        ent.gen += 1
        ent.consumed = False
        ent.node = _weak(ctx)
        ent.fwd.replay()
        model.last_masked_indices, model.last_unmasked_indices = ent.masked.clone(), ent.unmasked.clone()
        ctx.model, ctx.ent, ctx.gen, ctx.live = model, ent, ent.gen, live
        return ent.loss.reshape(()).clone()

    @staticmethod
    def backward(ctx, gout):
        ent, A = ctx.ent, ctx.model.arena
        if ctx.gen != ent.gen or ent.consumed:
            raise M3LError("backward through a CUDA-graph replayed forward whose saved activations were overwritten by a "
                           "newer forward of the same shape (or a second backward): set model.use_cuda_graph = False "
                           "for this pattern")
        ent.consumed = True
        ent.gout.copy_(gout.reshape(()))
        ent.bwd.replay()
        g = ent.gflat.clone()          # the static buffer is zeroed by the next replay; .grad must never alias it
        return (None, None, None, None, *[A.view(g, k) for k in ctx.live])


def _capture_emb_graphs(model, xs, geo, B):
    """Forward / backward graphs of get_embeddings (no-mask encoder pass), same scheme as _capture_mae_graphs."""
    A = model.arena
    ent = _GraphEntry()
    ent.xs = clone_inputs(xs)
    ent.gflat = A.new_grad_buffer()
    ent.gout = torch.zeros((B * geo.n, model.cfg.dim), dtype=torch.bfloat16, device=A.device)
    ent.gen, ent.consumed, ent.node = 0, True, None

    def fwd():
        out, ent.ctx = engine.embeddings_forward(model, ent.xs, geo, B, training=True)
        ent.loss = out.float().reshape(B, geo.n, model.cfg.dim)

    def bwd():
        ent.gflat.zero_()
        engine.embeddings_backward(model, ent.ctx, ent.gout, ent.gflat)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fwd()
        bwd()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    pool = torch.cuda.graph_pool_handle()
    ent.fwd, ent.bwd = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with engine.capture_guard():
        with torch.cuda.graph(ent.fwd, pool=pool):
            fwd()
        with torch.cuda.graph(ent.bwd, pool=pool):
            bwd()
    return ent


class _EmbGraphFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, ent, live, *params):
        ent.gen += 1
        ent.consumed = False
        ent.node = _weak(ctx)
        ent.fwd.replay()
        ctx.model, ctx.ent, ctx.gen, ctx.live = model, ent, ent.gen, live
        return ent.loss.clone()

    @staticmethod
    def backward(ctx, gout):
        ent, A = ctx.ent, ctx.model.arena
        if ctx.gen != ent.gen or ent.consumed:
            raise M3LError("backward through a CUDA-graph replayed get_embeddings whose saved activations were overwritten "
                           "by a newer call of the same shape (or a second backward): set model.use_cuda_graph = False")
        ent.consumed = True
        ent.gout.copy_(gout.reshape(ent.gout.shape))
        ent.bwd.replay()
        g = ent.gflat.clone()
        return (None, None, None, *[A.view(g, k) for k in ctx.live])


class _MAEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, xs, noise, geo, live, *params):
        need = any(ctx.needs_input_grad)
        gflat = model.arena.new_grad_buffer() if need else None
        loss_acc, c = engine.mae_forward(model, xs, noise, geo, training=need, gflat=gflat)
        ctx.model, ctx.c, ctx.live = model, c, live
        return loss_acc.reshape(())

    @staticmethod
    def backward(ctx, gout):
        model, A = ctx.model, ctx.model.arena
        # the buffer the forward pass put the head bias gradients into (first backward only)
        gflat = ctx.c.get("gflat_fwd")
        if gflat is None or ctx.c.get("gflat_used"):
            gflat = A.new_grad_buffer()
        ctx.c["gflat_used"] = True
        engine.mae_backward_decoder(model, ctx.c, gflat)
        engine.mae_backward_encoder(model, ctx.c, gflat)
        gflat.mul_(gout)
        return (None, None, None, None, None, *[A.view(gflat, k) for k in ctx.live])


class _EmbFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, xs, geo, B, live, *params):
        need = any(ctx.needs_input_grad)
        out, c = engine.embeddings_forward(model, xs, geo, B, training=need)
        ctx.model, ctx.c, ctx.live = model, c, live
        return out.float().reshape(B, geo.n, model.cfg.dim)

    @staticmethod
    def backward(ctx, gout):
        model, A = ctx.model, ctx.model.arena
        gflat = A.new_grad_buffer()
        dout = gout.reshape(-1, model.cfg.dim).to(torch.bfloat16).contiguous()
        engine.embeddings_backward(model, ctx.c, dout, gflat)
        return (None, None, None, None, None, *[A.view(gflat, k) for k in ctx.live])
