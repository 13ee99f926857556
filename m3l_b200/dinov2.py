"""DINOv2 ViT-S/14-with-registers image branch of the DINO-tac-MAE variant, on the kernel path, and the
feature extractor that concatenates its class token with the MAE latents.

Reference (paths under /root/reference):
  train_dino_tac_mae.py:29-31                       dino = torch.hub.load('facebookresearch/dinov2', 'dinov2_vits14_reg'); frozen
  models/pretrain_models_dino_cat_mae.py:792-841    MAEExtractor(observation_space, dino_model, mae_model, dim_embeddings, ...)
  models/pretrain_models_dino_cat_mae.py:866-904    forward: MAE latents -> vit_layer -> token mean, DINO class token of the
                                                    mid frame, cat, 3-layer mlp

`DinoV2` has the torch.hub model's constructor defaults, module tree and state_dict names, so
`DinoV2().load_state_dict(hub_model.state_dict())` works; its forward (frozen, no gradients, as the reference uses
it; differentiable for fine-tuning in training mode, see DinoV2) is a sequence of the C-ABI kernels: patchify (raw
observation or NCHW map) -> tcgen05 GEMM (patch embedding as a Linear over (p1, p2, c)-ordered patches) -> token
assembly (class / register tokens + position table) -> 12 x [LayerNorm, QKV GEMM, fused attention (6 heads x 64),
projection GEMM with LayerScale folded into its weights + residual, LayerNorm, FF1 GEMM + GELU, FF2 GEMM (LayerScale
folded) + residual] -> final LayerNorm of the class rows only.
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
    """dinov2_vits14_reg by default (embed_dim 384, depth 12, 6 heads, 4 register tokens, 37 x 37 position grid).

    Frozen or fine-tuned.  forward is differentiable with respect to the parameters when all three hold: grad mode
    is on, the module is in training mode (`.train()`), and at least one parameter other than `mask_token` has
    requires_grad.  Otherwise it runs the frozen sequence (no autograd, weights prepared once per version, forward
    replayed from a CUDA graph): an eval-mode module, or any call under torch.no_grad(), stays on it.  DINOv2 has no
    dropout or drop-path, so both paths compute the same function and return bit-identical outputs.

    Fine-tuning follows requires_grad: only trainable parameters receive a gradient (the others keep grad None),
    activations are kept only for blocks at or above the lowest block with a trainable parameter and the backward
    stops there, and the patch embedding / class, register and position tokens are differentiated only when one of
    them is trainable.  `mask_token` gets no gradient (the forward never reads it) and there is no gradient with
    respect to the input image.  Gradients accumulate into .grad as usual; step the parameters with any torch
    optimizer (the kernel operands are refreshed from them at every forward)."""

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

    def _token_table(self, gh, gw):
        """Additive (1 + R + gh*gw, D) fp32 table of the assembled tokens: class token + position 0, register tokens,
        patch positions."""
        pos = self._pos_table(gh, gw)
        return torch.cat([self.cls_token.detach().float()[0] + pos[:1], self.register_tokens.detach().float()[0],
                          pos[1:]], 0)

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
        add1 = self._token_table(gh, gw)
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
    use_cuda_graph = True        # replay the ~90-kernel forward (and the training backward) from CUDA graphs

    def forward(self, x, return_tokens: bool = False):
        """x: fp32 (B, 3, H, W) CUDA tensor, or a data.RawMap view of three channels of a raw observation.
        Returns the normalised class token (B, embed_dim) fp32 (what the hub model's forward returns), or with
        return_tokens=True all normalised tokens (B, 1 + R + H/14 * W/14, embed_dim).

        The output is differentiable with respect to the parameters when grad mode is on, the module is in training
        mode and at least one parameter other than `mask_token` has requires_grad (fine-tuning; see _forward_train).
        In every other case the frozen sequence runs without autograd: it is launch-bound at rollout /
        small-minibatch sizes (7 kernels per block behind Python + ctypes), so the kernel sequence is captured once
        per (batch, height, width) and replayed: the three input channels are first gathered into a static NCHW
        buffer (one `m3l_vt_load` launch, or a copy for tensor inputs).  DINOv2 has no dropout or drop-path, so both
        modes compute the same function."""
        if torch.is_grad_enabled() and self.training:
            live = [(k, p) for k, p in self.named_parameters() if p.requires_grad and k != "mask_token"]
            if live:
                return self._forward_train(x, return_tokens, live)
        return self._forward_frozen(x, return_tokens)

    @torch.no_grad()
    def _forward_frozen(self, x, return_tokens: bool = False):
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
        _load_input(x, static_in)
        g.replay()
        return out.clone()

    @torch.no_grad()
    def _forward_eager(self, x, return_tokens: bool = False):
        x = _as_source(x)
        B, C, H, W = x.shape
        assert C == 3, "DINOv2 takes three image channels"
        prep = self._prepare(H // self.patch_size, W // self.patch_size)
        return self._sequence(x, prep, return_tokens)

    def _rows(self, prep, B, n, dev):
        """Slot of every assembled token (-1: class / register token) and the output row of every class-token row."""
        slots = prep["slots"].get((B, n))
        if slots is None:
            R = self.num_register_tokens
            t = torch.arange(n, device=dev, dtype=torch.int32) - (1 + R)
            slots = prep["slots"][(B, n)] = torch.where(t >= 0, t, torch.full_like(t, -1)).repeat(B).contiguous()
            r = torch.arange(B * n, device=dev, dtype=torch.int32)
            prep["cls_rows"][(B, n)] = torch.where(r % n == 0, r // n, torch.full_like(r, -1)).contiguous()
        return slots, prep["cls_rows"][(B, n)]

    def _sequence(self, x, prep, return_tokens, saved: Optional[dict] = None):
        """The kernel sequence of the forward on the operands in `prep`.  saved (training): a dict with `lo` (lowest
        block whose activations the backward needs) and `emb` (whether it reaches the patch embedding); it receives
        the LayerNorm statistics, attention log-sum-exps, GELU' and the activations those blocks' backward reads."""
        B, C, H, W = x.shape
        ps, D, R, heads = self.patch_size, self.embed_dim, self.num_register_tokens, self.num_heads
        gh, gw = H // ps, W // ps
        npatch, n = gh * gw, 1 + R + gh * gw
        dev = prep["wpe"].device
        slots, cls_rows = self._rows(prep, B, n, dev)
        src = ops.make_patch_source([x], ps, ps, 0)
        cols = ops.patchify(src, B, npatch, ld=prep["ld"])
        tok = ops.gemm(cols, prep["wpe"], bias=prep["bpe"])
        xs = ops.decoder_assemble_fwd(tok, npatch, prep["zero"], slots, B, n, add1=prep["add1"])
        scale = 64 ** -0.5
        for i, blk in enumerate(prep["blocks"]):
            keep = saved is not None and i >= saved["lo"]
            y, st1 = ops.layernorm_fwd(xs, *blk["n1"], eps=1e-6, want_stats=keep)
            qkv = ops.gemm(y, blk["wqkv"], bias=blk["bqkv"])
            o, lse = ops.mha_fwd(qkv, B, n, heads, 64, scale)
            x_mid = ops.gemm(o, blk["wproj"], bias=blk["bproj"], residual=xs)
            y2, st2 = ops.layernorm_fwd(x_mid, *blk["n2"], eps=1e-6, want_stats=keep)
            pre = torch.empty((B * n, blk["w1"].shape[0]), dtype=torch.bfloat16, device=dev) if keep else None
            h = ops.gemm(y2, blk["w1"], bias=blk["b1"], act=ops.GELU_FWD, aux_out=pre)
            x_out = ops.gemm(h, blk["w2"], bias=blk["b2"], residual=x_mid)
            if keep:
                saved["blocks"].append((xs, y, st1, qkv, o, lse, x_mid, y2, st2, pre, h))
            xs = x_out
        train = saved is not None
        if return_tokens:
            out, st = ops.layernorm_fwd(xs, *prep["norm"], eps=1e-6, want_stats=train)
            res = out.float().reshape(B, n, D)
        else:
            out, st = ops.layernorm_fwd(xs, *prep["norm"], eps=1e-6, want_stats=train, out_rows=B, dst_row=cls_rows)
            res = out.float()
        if train:
            saved.update(xs=xs, st=st, B=B, gh=gh, gw=gw, n=n, npatch=npatch, slots=slots,
                         cls_rows=None if return_tokens else cls_rows, cols=cols if saved["emb"] else None)
        return res

    # ------------------------------------------------------------------ fine-tuning
    def _forward_train(self, x, return_tokens, live):
        """Differentiable forward: the frozen path's kernel sequence (bit-identical outputs) that also keeps what the
        backward reads, for the blocks at or above the lowest one with a trainable parameter (and the patchified
        input when the patch embedding / token tables are trainable).  The bf16 operands (LayerScale folded, plain
        and transposed) are refreshed in place from the parameters at the start of every forward, so an optimizer
        step between calls needs no re-capture.  Forward and backward replay from two CUDA graphs per
        (batch, height, width, trainable set, return_tokens)."""
        names = tuple(k for k, _ in live)
        params = [p for _, p in live]
        T = self._train_operands()
        plan = _TrainPlan(self, names)
        if not self.use_cuda_graph or torch.cuda.is_current_stream_capturing():
            step = _EagerStep(self, T, plan, _as_source(x), return_tokens)
        else:
            B, C, H, W = x.shape
            key = (B, H, W, names, bool(return_tokens))
            cache = T["graphs"]
            ent = cache.get(key)
            if ent is None:
                if len(cache) >= 4:
                    cache.pop(next(iter(cache)))
                ent = cache[key] = _capture_train(self, T, plan, B, H, W, return_tokens)
            _load_input(x, ent.static_in)
            step = _GraphStep(ent)
        return _TrainFn.apply(step, *params)

    def _train_operands(self):
        """bf16 / folded GEMM operands of the training path, allocated once per parameter storage and refreshed in
        place by _refresh (torch only allocates here)."""
        key = tuple(p.data_ptr() for p in self.parameters())
        T = self.__dict__.get("_train_ops")
        if T is not None and T["key"] == key:
            return T
        for k, p in self.named_parameters():
            if not p.is_cuda or p.dtype != torch.float32 or not p.is_contiguous():
                raise M3LError(f"m3l_b200.DinoV2 fine-tuning needs contiguous fp32 CUDA parameters ({k} is not; "
                               "no CPU fallback)")
        dev = self.cls_token.device
        D, P = self.embed_dim, 3 * self.patch_size ** 2
        ld = (P + 7) // 8 * 8
        bf = lambda *s: torch.empty(*s, dtype=torch.bfloat16, device=dev)
        T = {"key": key, "ld": ld, "wpe32": torch.zeros(D, ld, device=dev), "wpe": bf(D, ld),
             "bpe": self.patch_embed.proj.bias, "zero": torch.zeros(D, device=dev),
             "norm": (self.norm.weight, self.norm.bias), "blocks": [], "slots": {}, "cls_rows": {}, "graphs": {}}
        for b in self.blocks:
            hid = b.mlp.fc1.weight.shape[0]
            T["blocks"].append(dict(
                n1=(b.norm1.weight, b.norm1.bias), n2=(b.norm2.weight, b.norm2.bias),
                wqkv=bf(3 * D, D), wqkv_t=bf(D, 3 * D), bqkv=b.attn.qkv.bias,
                wproj=bf(D, D), wproj_t=bf(D, D), bproj=torch.empty(D, device=dev),
                w1=bf(hid, D), w1_t=bf(D, hid), b1=b.mlp.fc1.bias,
                w2=bf(D, hid), w2_t=bf(hid, D), b2=torch.empty(D, device=dev)))
        self.__dict__["_train_ops"] = T
        return T

    def _refresh(self, T, lo):
        """Rewrites the operands in T from the current parameter values (transposed copies for blocks >= lo only:
        the dgrad products of the backward read them)."""
        D, ps = self.embed_dim, self.patch_size
        P = 3 * ps * ps
        T["wpe32"][:, :P].copy_(self.patch_embed.proj.weight.detach().permute(0, 2, 3, 1).reshape(D, P))
        ops.cast_bf16(T["wpe32"], T["wpe"])
        for i, (b, tb) in enumerate(zip(self.blocks, T["blocks"])):
            tr = i >= lo
            ops.layerscale_fold(b.attn.qkv.weight, None, None, tb["wqkv"], tb["wqkv_t"] if tr else None)
            ops.layerscale_fold(b.attn.proj.weight, b.attn.proj.bias, b.ls1.gamma, tb["wproj"],
                                tb["wproj_t"] if tr else None, tb["bproj"])
            ops.layerscale_fold(b.mlp.fc1.weight, None, None, tb["w1"], tb["w1_t"] if tr else None)
            ops.layerscale_fold(b.mlp.fc2.weight, b.mlp.fc2.bias, b.ls2.gamma, tb["w2"], tb["w2_t"] if tr else None,
                                tb["b2"])

    def _train_fwd(self, T, plan, x, return_tokens):
        C = x.shape[1]
        assert C == 3, "DINOv2 takes three image channels"
        self._refresh(T, plan.lo)
        ps = self.patch_size
        prep = dict(T, add1=self._token_table(x.shape[2] // ps, x.shape[3] // ps))
        saved = {"lo": plan.lo, "emb": plan.emb, "blocks": [], "return_tokens": return_tokens}
        out = self._sequence(x, prep, return_tokens, saved)
        return out, saved

    def _train_bwd(self, T, saved, dout, G):
        """Backward of _train_fwd: dout bf16 (B or B*n rows, D) -> parameter gradients in the buffer G (zeroed).
        Per block in reverse, as engine.stack_bwd: FF2 (wgrad; its bias gradient is the column sum of dx, accumulated
        by the producer of dx), FF1 through GELU' (bias gradient in the dgrad epilogue), LayerNorm 2, projection,
        dO with the attention delta in its epilogue, attention, qkv (bias = column sum), LayerNorm 1; then the
        LayerScale unfold of the projection and FF2 gradients."""
        D, heads, R, ps = self.embed_dim, self.num_heads, self.num_register_tokens, self.patch_size
        depth, lo = len(self.blocks), saved["lo"]
        B, n = saved["B"], saved["n"]
        dx = ops.layernorm_bwd(dout, saved["xs"], saved["st"], self.norm.weight, dgamma=G("norm.weight"),
                               dbeta=G("norm.bias"), src_row=saved["cls_rows"],
                               dx_colsum=G(f"~{depth - 1}.db2") if lo < depth else None)
        fork = engine.WgradFork(dout.device)
        scale = 64 ** -0.5
        for l in reversed(range(lo, depth)):
            b, tb, p = self.blocks[l], T["blocks"][l], f"blocks.{l}."
            xs, y, st1, qkv, o, lse, x_mid, y2, st2, pre, h = saved["blocks"][l - lo]
            fork.wgrad(dx, h, G(f"~{l}.dw2"))
            dpre = ops.gemm(dx, tb["w2_t"], act=ops.GELU_BWD, aux_in=pre, colsum_out=G(p + "mlp.fc1.bias"))
            fork.wgrad(dpre, y2, G(p + "mlp.fc1.weight"))
            dx_mid = engine._dgrad_ln_bwd(dpre, tb["w1_t"], x_mid, st2, b.norm2.weight, G(p + "norm2.weight"),
                                          G(p + "norm2.bias"), dx, G(f"~{l}.dbp"))
            fork.wgrad(dx_mid, o, G(f"~{l}.dwp"))
            delta = torch.empty((B * n, heads), dtype=torch.float32, device=dx.device)
            do = ops.gemm(dx_mid, tb["wproj_t"], dot_side=o, dot_out=delta)
            dqkv = ops.mha_bwd(qkv, o, do, lse, B, n, heads, 64, scale, delta=delta)
            ops.colsum(dqkv, G(p + "attn.qkv.bias"))
            fork.wgrad(dqkv, y, G(p + "attn.qkv.weight"))
            dx_in = engine._dgrad_ln_bwd(dqkv, tb["wqkv_t"], xs, st1, b.norm1.weight, G(p + "norm1.weight"),
                                         G(p + "norm1.bias"), dx_mid, G(f"~{l - 1}.db2") if l > lo else None)
            fork.join()          # this block's wgrad operands (dx, dpre, dx_mid, dqkv) die below
            ops.layerscale_unfold(G(f"~{l}.dwp"), G(f"~{l}.dbp"), b.attn.proj.weight, b.attn.proj.bias, b.ls1.gamma,
                                  G(p + "attn.proj.weight"), G(p + "attn.proj.bias"), G(p + "ls1.gamma"))
            ops.layerscale_unfold(G(f"~{l}.dw2"), G(f"~{l}.db2"), b.mlp.fc2.weight, b.mlp.fc2.bias, b.ls2.gamma,
                                  G(p + "mlp.fc2.weight"), G(p + "mlp.fc2.bias"), G(p + "ls2.gamma"))
            dx = dx_in
        if not saved["emb"]:
            return
        # token assembly: patch-token gradient, and the (n, D) table gradient summed over the batch
        dtab = G("~dtab")
        dtok = ops.decoder_assemble_bwd(dx, saved["slots"], B, n, saved["npatch"], dadd1=dtab)
        ops.colsum(dtok, G("patch_embed.proj.bias"))
        engine.wgrad(dtok, saved["cols"], G("~dwpe"))
        P = 3 * ps * ps
        G("patch_embed.proj.weight").copy_(G("~dwpe")[:, :P].view(D, ps, ps, 3).permute(0, 3, 1, 2))
        G("cls_token").view(D).copy_(dtab[0])
        G("register_tokens").view(R, D).copy_(dtab[1:1 + R])
        gpos = G("pos_embed")[0]
        gpos[0].copy_(dtab[0])
        gpos[1:].copy_(pos_table_bwd(dtab[1 + R:], gpos.shape[0] - 1, saved["gh"], saved["gw"]))


def pos_table_bwd(dpatch, n_pos, gh, gw):
    """Gradient w.r.t. the patch rows (n_pos, D) of the position table from that w.r.t. the (gh*gw, D) rows
    DinoV2._pos_table made of them: identity when the grids match, else the backward of the antialiased bicubic
    resampling (parameter-sized, graph-capturable)."""
    if n_pos == gh * gw and gh == gw:
        return dpatch
    g = int(math.sqrt(n_pos))
    D = dpatch.shape[-1]
    d = dpatch.reshape(1, gh, gw, D).permute(0, 3, 1, 2).contiguous()
    d = torch.ops.aten._upsample_bicubic2d_aa_backward(d, [gh, gw], [1, D, g, g], False, None, None)
    return d.permute(0, 2, 3, 1).reshape(g * g, D)


def _as_source(x):
    """A tensor input as a layout-1 patch source (any strided NCHW view, e.g. a channel slice of the stacked image,
    with identity normalisation: no copy); a data.RawMap as it is."""
    if isinstance(x, RawMap):
        return x
    if not x.is_cuda:
        raise M3LError("m3l_b200.DinoV2: input is not on a CUDA device (no CPU fallback)")
    x = x.detach().to(torch.float32)
    B, C, H, W = x.shape
    return RawMap(x, (B, C, H, W), 0, x.stride(0), C, 0, x.stride(1), x.stride(2), x.stride(3), 0.0, 1.0,
                  strided_view=True)


def _load_input(x, static_in):
    """Gathers the input into the static NCHW buffer a captured graph reads."""
    if isinstance(x, RawMap):
        ops.vt_load_map(x, out=static_in)
    else:
        if not x.is_cuda:
            raise M3LError("m3l_b200.DinoV2: input is not on a CUDA device (no CPU fallback)")
        static_in.copy_(x, non_blocking=True)


_EMBED_PARAMS = ("patch_embed.proj.weight", "patch_embed.proj.bias", "cls_token", "register_tokens", "pos_embed")


class _TrainPlan:
    """What the backward of one trainable set covers: `lo`, the lowest block it runs (the lowest block with a
    trainable parameter; 0 when a token-embedding parameter is trainable, len(blocks) when only the final LayerNorm
    is), `emb`, whether it reaches the patch embedding and token tables, and the gradient buffer layout: the
    gradients of every parameter from block lo up (and of the embedding when emb), then fp32 scratch of the folded
    projection / FF2 weight gradients and of the embedding's intermediate products."""

    def __init__(self, model, live_names):
        depth = len(model.blocks)
        self.live = live_names
        self.emb = any(k in _EMBED_PARAMS for k in live_names)
        self.lo = 0 if self.emb else min((int(k.split(".")[1]) for k in live_names if k.startswith("blocks.")),
                                         default=depth)
        params = dict(model.named_parameters())
        names = (list(_EMBED_PARAMS) if self.emb else []) + \
            [k for k in params if k.startswith("blocks.") and int(k.split(".")[1]) >= self.lo] + ["norm.weight", "norm.bias"]
        self.layout = [(k, tuple(params[k].shape)) for k in names]
        D = model.embed_dim
        for l in range(self.lo, depth):
            hid = model.blocks[l].mlp.fc1.weight.shape[0]
            self.layout += [(f"~{l}.dwp", (D, D)), (f"~{l}.dbp", (D,)), (f"~{l}.dw2", (D, hid)), (f"~{l}.db2", (D,))]
        self.n_params = len(names)

    def grads(self, device, n, ld, D):
        layout = self.layout + ([("~dwpe", (D, ld)), ("~dtab", (n, D))] if self.emb else [])
        return _GradBuffer(layout, self.n_params, device)


class _GradBuffer:
    """One zeroed fp32 buffer holding the entries of a _TrainPlan layout (64-element aligned)."""

    def __init__(self, layout, n_params, device):
        self.off, off = {}, 0
        for i, (k, shape) in enumerate(layout):
            if i == n_params:
                self.params_end = off
            self.off[k] = (off, shape)
            off += (math.prod(shape) + 63) // 64 * 64
        if n_params == len(layout):
            self.params_end = off
        self.flat = torch.zeros(off, dtype=torch.float32, device=device)

    def __call__(self, k, flat=None):
        o, shape = self.off[k]
        return (self.flat if flat is None else flat)[o:o + math.prod(shape)].view(shape)

    def hand_out(self, names, clone: bool):
        """The gradients of `names`, as views of one copy of the parameter region when clone (a static buffer that
        the next replay overwrites must never be aliased by .grad)."""
        flat = self.flat[:self.params_end].clone() if clone else self.flat
        return [self(k, flat) for k in names]


class _EagerStep:
    """One training forward / backward issued kernel by kernel (use_cuda_graph = False, or inside a capture)."""

    def __init__(self, model, T, plan, x, return_tokens):
        self.model, self.T, self.plan, self.x, self.return_tokens = model, T, plan, x, return_tokens

    def forward(self):
        self.out, self.saved = self.model._train_fwd(self.T, self.plan, self.x, self.return_tokens)
        return self.out

    def backward(self, gout):
        m, s = self.model, self.saved
        G = self.plan.grads(gout.device, s["n"], self.T["ld"], m.embed_dim)
        dout = gout.reshape(-1, m.embed_dim).to(torch.bfloat16).contiguous()
        m._train_bwd(self.T, s, dout, G)
        return G.hand_out(self.plan.live, clone=False)


class _TrainEntry:
    __slots__ = ("fwd", "bwd", "static_in", "out", "saved", "G", "gout", "live", "gen", "consumed")


def _capture_train(model, T, plan, B, H, W, return_tokens):
    """Forward / backward CUDA graphs of one (batch, size, trainable set, return_tokens), sharing one memory pool
    (the forward graph's saved activations are the backward graph's inputs), as vtmae._capture_mae_graphs."""
    dev = T["wpe"].device
    D, ps = model.embed_dim, model.patch_size
    n = 1 + model.num_register_tokens + (H // ps) * (W // ps)
    ent = _TrainEntry()
    ent.static_in = torch.zeros((B, 3, H, W), dtype=torch.float32, device=dev)
    ent.G = plan.grads(dev, n, T["ld"], D)
    ent.gout = torch.zeros((B * n if return_tokens else B, D), dtype=torch.bfloat16, device=dev)
    ent.live, ent.gen, ent.consumed = plan.live, 0, True
    src = _as_source(ent.static_in)

    def fwd():
        ent.out, ent.saved = model._train_fwd(T, plan, src, return_tokens)

    def bwd():
        ent.G.flat.zero_()
        model._train_bwd(T, ent.saved, ent.gout, ent.G)

    with torch.no_grad():
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):                   # warm-up: lazy tables, kernel attributes, allocator
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


class _GraphStep:
    """One training forward / backward replayed from a _TrainEntry."""

    def __init__(self, ent):
        self.ent = ent

    def forward(self):
        ent = self.ent
        ent.gen += 1
        ent.consumed = False
        self.gen = ent.gen
        ent.fwd.replay()
        return ent.out.clone()

    def backward(self, gout):
        ent = self.ent
        if self.gen != ent.gen or ent.consumed:
            raise M3LError("backward through a CUDA-graph replayed DinoV2 forward whose saved activations were "
                           "overwritten by a newer forward of the same shape (or a second backward): set "
                           "model.use_cuda_graph = False for this pattern")
        ent.consumed = True
        ent.gout.copy_(gout.reshape(ent.gout.shape))
        ent.bwd.replay()
        return ent.G.hand_out(ent.live, clone=True)


class _TrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, step, *params):
        ctx.step = step
        return step.forward()

    @staticmethod
    def backward(ctx, gout):
        return (None, *ctx.step.backward(gout.contiguous()))


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
        with torch.no_grad():                                                     # frozen whatever the module mode
            cls = self.dino_model(mid_frame_view(views['image'], self.frame_stack))  # (B, dim)
        return self.mlp(torch.cat((latents, cls.to(latents.dtype)), dim=-1))
