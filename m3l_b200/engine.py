"""Host-side sequencing of the CUDA kernels for the VTMAE step (forward, backward) and for the
no-mask encoder pass.  Pure plumbing: every arithmetic step is a C-ABI kernel call (m3l_b200.ops);
torch only allocates buffers and provides the stream, so the whole sequence can be captured in a
CUDA graph (m3l_b200.trainer).

Reference semantics followed (paths relative to /root/reference):
  VTMAE.forward          models/pretrain_models.py:146-342   (early_conv_masking=False path)
  VTMAE.get_embeddings   models/pretrain_models.py:588-668
  vit_pytorch Transformer (pre-norm attention + feed-forward blocks, final LayerNorm): SURVEY.md A.2
"""
from __future__ import annotations

import contextlib
import gc
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch

from . import ops
from .arena import ParamArena

import os

_SM_COUNT_CACHE = {}


def _sm_count() -> int:
    """SMs of the current device (148 on B200; MIG slices and other SKUs differ): sizes the single-wave wgrad tiling."""
    dev = torch.cuda.current_device() if torch.cuda.is_available() else -1
    n = _SM_COUNT_CACHE.get(dev)
    if n is None:
        n = _SM_COUNT_CACHE[dev] = torch.cuda.get_device_properties(dev).multi_processor_count if dev >= 0 else 148
    return n
# M3L_FUSED_MLP=0: the unfused LayerNorm / FF1+GELU / FF2 kernels instead of csrc/rowblock.cu (A/B measurements)
_FUSED_MLP = os.environ.get("M3L_FUSED_MLP", "1") != "0"
# M3L_FUSED_LN_BWD=0: separate dgrad GEMM + LayerNorm-backward kernels instead of the GEMM's fused epilogue (A/B measurements)
_FUSED_LN_BWD = os.environ.get("M3L_FUSED_LN_BWD", "1") != "0"
# the fused epilogue needs BN = 256 tiles of 128 full rows: below this many rows the tiles no longer cover the SMs (the
# encoder's 2560 rows are 20 tiles: measured 207 -> 247 us for the encoder backward) and the two separate kernels win
_FUSED_LN_BWD_MIN_ROWS = int(os.environ.get("M3L_FUSED_LN_BWD_MIN_ROWS", "16384"))


def _dgrad_ln_bwd(dy_in, w_t, x, stats, gamma, dgamma, dbeta, skip, dx_colsum):
    """dx = dLN(dy_in @ w_t.T; x, stats, gamma) + skip, with the LayerNorm parameter gradients and the column sums of
    dx accumulated: one GEMM with the LayerNorm backward in its epilogue when the normalised dimension is 256 (the
    gradient w.r.t. the LayerNorm output never reaches HBM), else the dgrad GEMM followed by the LayerNorm-backward kernel."""
    if _FUSED_LN_BWD and x.shape[1] == 256 and x.shape[0] >= _FUSED_LN_BWD_MIN_ROWS:
        return ops.gemm(dy_in, w_t, ln_bwd=dict(x=x, stats=stats, gamma=gamma, skip=skip, dgamma=dgamma, dbeta=dbeta,
                                               dx_colsum=dx_colsum))
    dxn = ops.gemm(dy_in, w_t)
    return ops.layernorm_bwd(dxn, x, stats, gamma, dgamma=dgamma, dbeta=dbeta, skip=skip, dx_colsum=dx_colsum)


@dataclass
class StackSpec:
    prefix: str
    dim: int
    depth: int
    heads: int
    dim_head: int
    mlp_dim: int

    @property
    def inner(self):
        return self.heads * self.dim_head


def _wgrad_tiling(m_out: int, n_out: int, k_tokens: int):
    """(BN, split-K) for a wgrad product: the widest N tile that divides n_out and as many splits as
    keep the whole problem in ONE wave of CTAs (measured best on B200: tools/sweep_wgrad.py)."""
    bn = 256 if n_out % 256 == 0 else (128 if n_out % 128 == 0 else 64)
    tiles = ((m_out + 127) // 128) * ((n_out + bn - 1) // bn)
    kb = (k_tokens + 63) // 64
    s = max(1, _sm_count() // tiles)
    return bn, max(1, min(s, kb))


def wgrad(dy: torch.Tensor, x: torch.Tensor, gview: torch.Tensor) -> None:
    """gview[out, in] += dy[M, out]^T @ x[M, in]  (split-K over the token rows, fp32 red.add)."""
    out_f, in_f = gview.shape
    bn, splits = _wgrad_tiling(out_f, in_f, dy.shape[0])
    ops.gemm(dy, x, mn_major=True, out=gview, accumulate=True, splits=splits, bn=bn)


@contextlib.contextmanager
def capture_guard():
    """Around a CUDA-graph capture: no cyclic-garbage collection inside it.  A stale model that owns captured graphs
    (e.g. one dropped by the caller but still in a reference cycle) would otherwise be finalised in the middle of the
    capture, and CUDAGraph.reset() / cudaFree are illegal while a stream is capturing."""
    gc.collect()
    torch.cuda.synchronize()
    was = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if was:
            gc.enable()


_SIDE_STREAMS: Dict = {}


def side_stream(device, index: int = 0) -> "torch.cuda.Stream":
    """Second stream for the weight-gradient GEMMs: they only feed the gradient arena, so they run
    beside the dgrad chain (the critical path) instead of inside it.  Forks/joins are event based and
    are captured as parallel branches of the CUDA graph."""
    key = (device.type, device.index, index)
    st = _SIDE_STREAMS.get(key)
    if st is None:
        st = torch.cuda.Stream(device=device)
        _SIDE_STREAMS[key] = st
    return st


class Branch:
    """Second, parallel branch of the kernel sequence (captured as a parallel branch of the CUDA graph): the image
    and the tactile halves of the patch embedding and of the reconstruction heads are independent chains of
    small, latency-bound kernels, so they run side by side instead of back to back.

        br = Branch(device)
        with br:            # kernels issued here go to the side stream, ordered after everything issued so far
            ...
        ...                 # main-stream work that does not depend on the branch
        br.join()           # main stream waits for the branch

    Buffers used inside the branch are allocated BEFORE entering it (main stream) and stay referenced until
    after join(), so the caching allocator never hands them to the other stream early."""

    def __init__(self, device, enabled: bool = True, index: int = 1):
        self.enabled = enabled
        self.main = torch.cuda.current_stream(device)
        self.side = side_stream(device, index) if enabled else None
        self._ctx = None

    def __enter__(self):
        if self.enabled:
            self.side.wait_stream(self.main)
            self._ctx = torch.cuda.stream(self.side)
            self._ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.enabled:
            self._ctx.__exit__(*exc)
        return False

    def join(self):
        if self.enabled:
            self.main.wait_stream(self.side)


class WgradFork:
    """Runs wgrad GEMMs on the side stream; join() before their operands may be freed or reused."""

    def __init__(self, device, enabled: bool = True):
        self.enabled = enabled
        self.main = torch.cuda.current_stream(device)
        self.side = side_stream(device) if enabled else None
        self.dirty = False

    def wgrad(self, dy, x, gview):
        if not self.enabled:
            wgrad(dy, x, gview)
            return
        self.side.wait_stream(self.main)
        with torch.cuda.stream(self.side):
            wgrad(dy, x, gview)
        self.dirty = True

    def join(self):
        if self.enabled and self.dirty:
            self.main.wait_stream(self.side)
            self.dirty = False


class GradView:
    """Accessor of per-parameter views into a flat fp32 gradient buffer laid out like the arena."""

    def __init__(self, arena: ParamArena, flat: torch.Tensor):
        self.arena, self.flat = arena, flat

    def __call__(self, name: str) -> torch.Tensor:
        return self.arena.view(self.flat, name)


# --------------------------------------------------------------------------------------------
# transformer stack (vit_pytorch.vit.Transformer without its final LayerNorm)
# --------------------------------------------------------------------------------------------
def p_drop(transformer) -> float:
    """Dropout probability in force for a transformer module (vtmae.Transformer): its `dropout` in training mode,
    0 in eval mode, as for the nn.Dropout layers of the reference."""
    return float(transformer.p_drop) if transformer.training else 0.0


def draw_dropout_key(device) -> torch.Tensor:
    """The key of the dropout masks of one stack_fwd call: int64 [1] drawn on the device from torch's default CUDA
    generator, so torch.manual_seed governs eager runs and every CUDA-graph replay draws a fresh key."""
    return torch.randint(0, 2 ** 62, (1,), dtype=torch.int64, device=device)


class _StackDropout:
    """The dropout of one stack_fwd call (probability p, one key for every layer and site), kept with the saved
    activations for stack_bwd."""

    def __init__(self, key: torch.Tensor, p: float):
        self.key, self.p = key, p

    def __call__(self, layer: int, site: int) -> "ops.Dropout":
        return ops.Dropout(self.key, (layer << 2) | site, self.p)


def stack_fwd(A: ParamArena, spec: StackSpec, x: torch.Tensor, B: int, n: int, saved: Optional[list],
              p_drop: float = 0.0):
    """x: bf16 [B*n, dim].  Returns the residual stream after the last block.
    p_drop > 0: vit_pytorch's four Dropout sites per layer (attention probabilities, to_out, after GELU, feed-forward
    output) with the masks of csrc/dropout.cuh under a key from draw_dropout_key; callers pass their training-mode
    probability, and 0 in eval mode.  The feed-forward block then runs as LayerNorm, GEMM + GELU, GEMM + residual,
    and attention through the dropout kernels at every length."""
    scale = spec.dim_head ** -0.5
    M = x.shape[0]
    drop = _StackDropout(draw_dropout_key(x.device), float(p_drop)) if p_drop > 0 else None
    for l in range(spec.depth):
        pa, pf = f"{spec.prefix}.layers.{l}.0", f"{spec.prefix}.layers.{l}.1"
        xn1, st1 = ops.layernorm_fwd(x, A.f32(pa + ".norm.weight"), A.f32(pa + ".norm.bias"),
                                     want_stats=saved is not None)
        qkv = ops.gemm(xn1, A.bf(pa + ".to_qkv.weight"))
        o, lse = ops.mha_fwd(qkv, B, n, spec.heads, spec.dim_head, scale, dropout=drop(l, 0) if drop else None)
        fused = _FUSED_MLP and ops.ln_mlp_supported(spec.dim, spec.mlp_dim) and drop is None
        # training keeps x_mid for the backward pass, so the attention-output GEMM writes its result twice (x_mid and
        # the buffer the fused feed-forward block then accumulates into); inference updates x_mid in place
        x_out = torch.empty_like(x) if (fused and saved is not None) else None
        x_mid = ops.gemm(o, A.bf(pa + ".to_out.0.weight"), bias=A.f32(pa + ".to_out.0.bias"), residual=x, out2=x_out,
                         dropout=drop(l, 1) if drop else None)
        if fused:
            # LayerNorm -> Linear -> GELU -> Linear -> + residual in ONE kernel; the [M, mlp_dim] hidden stays in
            # tensor memory (training additionally stores what the backward pass reads)
            r = ops.ln_mlp_fwd(x_mid, A.f32(pf + ".net.0.weight"), A.f32(pf + ".net.0.bias"),
                               A.bf(pf + ".net.1.weight"), A.f32(pf + ".net.1.bias"),
                               A.bf(pf + ".net.4.weight"), A.f32(pf + ".net.4.bias"), save=saved is not None,
                               out=x_out if saved is not None else x_mid, out_has_x=saved is not None)
            if saved is not None:
                x_out, st2, xn2, h, pre = r
            else:
                x_out, st2, xn2, h, pre = r, None, None, None, None
        else:
            xn2, st2 = ops.layernorm_fwd(x_mid, A.f32(pf + ".net.0.weight"), A.f32(pf + ".net.0.bias"),
                                         want_stats=saved is not None)
            pre = torch.empty((M, spec.mlp_dim), dtype=torch.bfloat16, device=x.device) if saved is not None else None
            h = ops.gemm(xn2, A.bf(pf + ".net.1.weight"), bias=A.f32(pf + ".net.1.bias"), act=ops.GELU_FWD, aux_out=pre,
                         dropout=drop(l, 2) if drop else None)
            x_out = ops.gemm(h, A.bf(pf + ".net.4.weight"), bias=A.f32(pf + ".net.4.bias"), residual=x_mid,
                             dropout=drop(l, 3) if drop else None)
        if saved is not None:
            saved.append((x, xn1, st1, qkv, o, lse, x_mid, xn2, st2, pre, h, drop))
        x = x_out
    return x


def last_ff_bias(spec: StackSpec) -> str:
    """Name of the bias whose gradient is the column sum of the stack-output gradient (without dropout)."""
    return f"{spec.prefix}.layers.{spec.depth - 1}.1.net.4.bias"


def stack_dx_colsum(G: GradView, spec: StackSpec, saved: list) -> Optional[torch.Tensor]:
    """Where the producer of stack_bwd's dx accumulates the column sums of dx: the gradient of the last feed-forward
    bias, G(last_ff_bias(spec)).  None when the forward applied dropout: that gradient is then the column sum of the
    dropped-out dx, which stack_bwd accumulates itself."""
    return None if saved[-1][-1] is not None else G(last_ff_bias(spec))


def stack_bwd(A: ParamArena, G: GradView, spec: StackSpec, dx: torch.Tensor, B: int, n: int, saved: list):
    """dx: bf16 [B*n, dim] gradient w.r.t. the stack output.  Returns the gradient w.r.t. its input.
    The producer of dx (the final-LayerNorm backward) must already have accumulated its column sums
    into stack_dx_colsum(G, spec, saved) when that is not None (dx_colsum= of ops.layernorm_bwd)."""
    scale = spec.dim_head ** -0.5
    M = dx.shape[0]
    fork = WgradFork(A.device)
    for l in reversed(range(spec.depth)):
        pa, pf = f"{spec.prefix}.layers.{l}.0", f"{spec.prefix}.layers.{l}.1"
        x, xn1, st1, qkv, o, lse, x_mid, xn2, st2, pre, h, drop = saved[l]
        # ---- feed-forward branch: x_out = x_mid + Z3 o (W2 h + b2), h = Z2 o gelu(W1 LN2(x_mid) + b1) (Z = 1 without
        # dropout); pre holds Z2 o gelu', so the GELU' product below is the backward through Z2 as well
        dy = dx
        if drop is not None:
            dy = ops.dropout_bwd(dx, drop(l, 3), colsum=G(pf + ".net.4.bias"))
        fork.wgrad(dy, h, G(pf + ".net.4.weight"))
        dpre = ops.gemm(dy, A.bf_t(pf + ".net.4.weight"), act=ops.GELU_BWD, aux_in=pre,
                        colsum_out=G(pf + ".net.1.bias"))
        fork.wgrad(dpre, xn2, G(pf + ".net.1.weight"))
        dx_mid = _dgrad_ln_bwd(dpre, A.bf_t(pf + ".net.1.weight"), x_mid, st2, A.f32(pf + ".net.0.weight"),
                               G(pf + ".net.0.weight"), G(pf + ".net.0.bias"), dx,
                               G(pa + ".to_out.0.bias") if drop is None else None)
        # ---- attention branch: x_mid = x + Z1 o (Wo attn(Wqkv LN1(x)) + bo), attention probabilities dropped by Z0
        dy_mid = dx_mid
        if drop is not None:
            dy_mid = ops.dropout_bwd(dx_mid, drop(l, 1), colsum=G(pa + ".to_out.0.bias"))
        fork.wgrad(dy_mid, o, G(pa + ".to_out.0.weight"))
        # dO, and in the same epilogue delta = rowsum(dO * O) per head (dim_head == 64 == one epilogue round)
        delta = torch.empty((M, spec.heads), dtype=torch.float32, device=dx.device) if spec.dim_head == 64 else None
        do = ops.gemm(dy_mid, A.bf_t(pa + ".to_out.0.weight"), dot_side=o if delta is not None else None, dot_out=delta)
        dqkv = ops.mha_bwd(qkv, o, do, lse, B, n, spec.heads, spec.dim_head, scale, delta=delta,
                           dropout=drop(l, 0) if drop else None)
        fork.wgrad(dqkv, xn1, G(pa + ".to_qkv.weight"))
        prev_bias = G(f"{spec.prefix}.layers.{l - 1}.1.net.4.bias") if (l > 0 and drop is None) else None
        dx_in = _dgrad_ln_bwd(dqkv, A.bf_t(pa + ".to_qkv.weight"), x, st1, A.f32(pa + ".norm.weight"),
                              G(pa + ".norm.weight"), G(pa + ".norm.bias"), dx_mid, prev_bias)
        fork.join()          # this layer's wgrad operands (dy, dpre, dy_mid, dqkv) die below
        dx = dx_in
    return dx


# --------------------------------------------------------------------------------------------
# geometry of one call (which modalities are present)
# --------------------------------------------------------------------------------------------
@dataclass
class Geometry:
    use_vision: bool
    nt: int                      # tactile sensors present in this call
    n_img: int
    n_tac: int                   # per sensor
    nm_img: int
    nm_tac: int                  # per sensor
    segs: List[Tuple[int, int, int]] = field(default_factory=list)

    @property
    def n(self):
        return self.n_img + self.nt * self.n_tac

    @property
    def nv_img(self):
        return self.n_img - self.nm_img

    @property
    def nv_tac(self):            # all sensors
        return self.nt * (self.n_tac - self.nm_tac)

    @property
    def nv(self):
        return self.nv_img + self.nv_tac

    @property
    def nm_tac_total(self):
        return self.nt * self.nm_tac

    @property
    def nm(self):
        return self.nm_img + self.nm_tac_total


def make_geometry(cfg, use_vision: bool, use_tactile: bool, reconstruct_ratio: Optional[float] = None) -> Geometry:
    nt = cfg.num_tactiles if (cfg.num_tactiles > 0 and use_tactile) else 0
    n_img = cfg.n_img if use_vision else 0
    n_tac = cfg.n_tac if nt else 0
    n = n_img + nt * n_tac
    if reconstruct_ratio is None:
        # Python-float truncations exactly as pretrain_models.py:223-227
        num_masked = int(cfg.masking_ratio * n)
        nm_img = int(num_masked * (n_img / n))
        nm_tac = (num_masked - nm_img) // cfg.num_tactiles if nt else 0
    else:
        # reconstruct() splits per modality instead (pretrain_models.py:425,433)
        nm_img = int(reconstruct_ratio * n_img) if n_img else 0
        nm_tac = int(reconstruct_ratio * (nt * n_tac) / cfg.num_tactiles) if nt else 0
    segs = ([(0, n_img, nm_img)] if n_img else []) + [(n_img + i * n_tac, n_tac, nm_tac) for i in range(nt)]
    return Geometry(use_vision, nt, n_img, n_tac, nm_img, nm_tac, segs)


class Tables:
    """Static per-(geometry, batch) index tables and additive position tables (device tensors)."""

    def __init__(self, model, geo: Geometry, B: int, device):
        cfg = model.cfg
        i32 = dict(dtype=torch.int32, device=device)
        self.B = B
        # token class (modality) per present token and per visible slot
        cls = [0] * geo.n_img + [1 + i for i in range(geo.nt) for _ in range(geo.n_tac)]
        self.tok_class = torch.tensor(cls, **i32)
        nv_t = geo.n_tac - geo.nm_tac
        slot_cls = [0] * geo.nv_img + [1 + i for i in range(geo.nt) for _ in range(nv_t)]
        self.slot_class = torch.tensor(slot_cls if slot_cls else [0], **i32)
        # masked path: embedding rows -> encoder rows
        b = torch.arange(B, device=device)[:, None]
        self.enc_dst_img = (b * geo.nv + torch.arange(geo.nv_img, device=device)[None]).reshape(-1).to(torch.int32)
        self.enc_dst_tac = (b * geo.nv + geo.nv_img + torch.arange(geo.nv_tac, device=device)[None]).reshape(-1).to(torch.int32)
        self.enc_cls_img = torch.zeros(B * geo.nv_img, **i32)
        self.enc_cls_tac = torch.tensor(slot_cls[geo.nv_img:] * B if geo.nv_tac else [0], **i32)
        # all-token path (get_embeddings)
        self.all_dst_img = (b * geo.n + torch.arange(geo.n_img, device=device)[None]).reshape(-1).to(torch.int32)
        self.all_dst_tac = (b * geo.n + geo.n_img + torch.arange(geo.nt * geo.n_tac, device=device)[None]).reshape(-1).to(torch.int32)
        self.all_cls_img = torch.zeros(max(B * geo.n_img, 1), **i32)
        self.all_cls_tac = torch.tensor((cls[geo.n_img:] * B) if geo.nt else [0], **i32)
        self.all_pos_img = torch.arange(geo.n_img, device=device).repeat(B).to(torch.int32)
        self.all_pos_tac = (geo.n_img + torch.arange(geo.nt * geo.n_tac, device=device)).repeat(B).to(torch.int32)
        # early_conv_masking: the heads run on ALL tokens; row of token (b, t) in the stacked head inputs
        # [B*n_img image rows | B*nt*n_tac tactile rows]
        t = torch.arange(geo.n, device=device)[None]
        nta = geo.nt * geo.n_tac
        img_row = b * geo.n_img + t
        tac_row = B * geo.n_img + b * nta + (t - geo.n_img)
        self.head_row_all = torch.where(t < geo.n_img, img_row, tac_row).reshape(-1).to(torch.int32)
        # sin-cos tables of the present tokens (constants, fp32)
        if cfg.use_sincosmod_encodings:
            enc, dec = [], []
            if geo.use_vision:
                enc.append(model.image_enc_pos_embedding[0]); dec.append(model.image_dec_pos_embedding[0])
            if geo.nt:
                k = geo.nt * geo.n_tac
                enc.append(model.tactile_enc_pos_embedding[0, :k]); dec.append(model.tactile_dec_pos_embedding[0, :k])
            self.enc_pos = torch.cat(enc, 0).to(device=device, dtype=torch.float32).contiguous()
            self.dec_pos = torch.cat(dec, 0).to(device=device, dtype=torch.float32).contiguous()
        else:
            self.enc_pos = self.dec_pos = None


# --------------------------------------------------------------------------------------------
# EarlyCNN conv stem (early_conv_masking=True; pretrain_models.py:37-56,180-191): im2col + GEMM
# --------------------------------------------------------------------------------------------
def cnn_layers(model, key: str):
    """[(name, cin, cout, k, stride, pad)] of EarlyCNN(key) (pretrain_models.py:41-49)."""
    cnn = model.early_conv_vision if key == "image" else model.early_conv_tactile
    out = []
    for nm in ("conv1", "conv2", "conv3", "conv4"):
        c = getattr(cnn, nm)
        out.append((nm, c.in_channels, c.out_channels, c.kernel_size[0], c.stride[0], c.padding[0]))
    return out


def _cnn_fwd(A, prefix: str, layers, maps: List[torch.Tensor], B: int, H: int, W: int, saved: Optional[list]):
    """maps: fp32 NCHW [B, C, H, W], one per source (the sensors of a modality share the CNN and are stacked
    along the batch).  Returns the tokens bf16 [len(maps)*B*h*w, D] in (source, sample, y, x) row order."""
    beff = B * len(maps)
    x, h, w = None, H, W
    for li, (nm, cin, cout, k, st, pd) in enumerate(layers):
        ho, wo = ops.conv_out_size(h, k, st, pd), ops.conv_out_size(w, k, st, pd)
        if li == 0:
            col = torch.empty((beff * ho * wo, cin * k * k), dtype=torch.bfloat16, device=A.device)
            for si, m in enumerate(maps):
                ops.im2col(m, B, cin, h, w, k, st, pd, False, out=col[si * B * ho * wo:(si + 1) * B * ho * wo])
        elif k == 1 and st == 1 and pd == 0:
            col = x                                         # 1x1 convolution: the activation matrix itself
        else:
            col = ops.im2col(x, beff, cin, h, w, k, st, pd, True)
        y = ops.gemm(col, A.bf2d(f"{prefix}.{nm}.weight"), bias=A.f32(f"{prefix}.{nm}.bias"),
                     act=ops.RELU if li < len(layers) - 1 else 0)
        if saved is not None:
            saved.append((col, y, h, w))
        x, h, w = y, ho, wo
    return x


def _cnn_bwd(A, G, prefix: str, layers, dtok: torch.Tensor, saved: list, beff: int):
    """dtok: bf16 gradient w.r.t. the conv-stem tokens (rows as _cnn_fwd returns them)."""
    dy = dtok
    for li in reversed(range(len(layers))):
        nm, cin, cout, k, st, pd = layers[li]
        col, y, h, w = saved[li]
        ops.colsum(dy, G(f"{prefix}.{nm}.bias"))
        wgrad(dy, col, G(f"{prefix}.{nm}.weight").view(cout, cin * k * k))
        if li == 0:
            break                                           # the raw maps need no gradient
        dcol = ops.gemm(dy, A.bf_t(f"{prefix}.{nm}.weight"))
        dy = ops.col2im_relu(dcol, beff, cin, h, w, k, st, pd, relu_out=saved[li - 1][1])


def _modalities(model, geo, x):
    """(key, prefix, maps, H, W, n_per_source, tok_base) of the modalities present."""
    e = model.encoder
    out = []
    mat = lambda t: t.materialize() if hasattr(t, "materialize") else t      # the conv stem reads NCHW maps
    if geo.use_vision:
        out.append(("image", "early_conv_vision", [mat(x["image"])], e.image_height, e.image_width, geo.n_img, 0))
    if geo.nt:
        out.append(("tactile", "early_conv_tactile", [mat(x[f"tactile{i + 1}"]) for i in range(geo.nt)],
                    e.tactile_height, e.tactile_width, geo.n_tac, geo.n_img))
    return out


def _embed_fwd_ecm(model, A, geo, tabs, x, B, masked: bool, saved: Optional[dict], unmasked32=None):
    """Encoder input rows from the conv stems (+ modality + position), visible tokens only when masked."""
    cfg = model.cfg
    D = cfg.dim
    n_rows = geo.nv if masked else geo.n
    x0 = torch.empty((B * n_rows, D), dtype=torch.bfloat16, device=A.device)
    sincos = cfg.use_sincosmod_encodings
    for key, prefix, maps, H, W, n_per, tok_base in _modalities(model, geo, x):
        layers = cnn_layers(model, key)
        cs = [] if saved is not None else None
        tok = _cnn_fwd(A, prefix, layers, maps, B, H, W, cs)
        img = key == "image"
        if masked:
            ncols, col0 = (geo.nv_img, 0) if img else (geo.nv_tac, geo.nv_img)
            dst = tabs.enc_dst_img if img else tabs.enc_dst_tac
        else:
            ncols, col0 = n_per * len(maps), 0
            dst = tabs.all_dst_img if img else tabs.all_dst_tac
        ops.token_finish(tok, B, n_per, ncols, tok_base, x0, tok_idx=unmasked32 if masked else None, col0=col0,
                         add0=A.f32("encoder_modality_embedding.weight") if sincos else None,
                         tok_class=tabs.tok_class if sincos else None,
                         add1=tabs.enc_pos if sincos else A.f32("encoder.pos_embedding")[0, 1:geo.n + 1], dst_row=dst)
        if saved is not None:
            saved[key] = (cs, layers, len(maps), n_per, tok_base)
    return x0


def _embed_bwd_ecm(model, A, G, geo, tabs, dx0, B, masked: bool, saved: dict, slots=None):
    cfg = model.cfg
    n_rows = geo.nv if masked else geo.n
    if cfg.use_sincosmod_encodings:
        ops.rowclass_sum(dx0, B, n_rows, slot_class=tabs.slot_class if masked else tabs.tok_class,
                         dclass=G("encoder_modality_embedding.weight"))
    else:
        gpos = G("encoder.pos_embedding")[0, 1:geo.n + 1]
        pos = saved["unmasked32"].view(-1) if masked else torch.arange(geo.n, device=dx0.device, dtype=torch.int32).repeat(B)
        ops.rowclass_sum(dx0, B, n_rows, row_pos=pos, dpos=gpos)
    for key in ("image", "tactile"):
        if key not in saved:
            continue
        cs, layers, nsrc, n_per, tok_base = saved[key]
        prefix = "early_conv_vision" if key == "image" else "early_conv_tactile"
        dtok = ops.token_finish_bwd(dx0, B, n_rows, geo.n, tok_base, nsrc * n_per, n_per,
                                    slot_of_token=slots if masked else None)
        _cnn_bwd(A, G, prefix, layers, dtok, cs, B * nsrc)


# --------------------------------------------------------------------------------------------
# token embedding:  LN(P) -> Linear -> LN(D) (+ modality + position)   [early_conv_masking=False]
# --------------------------------------------------------------------------------------------
def _embed_fwd(model, A, geo, tabs, x, B, tok_idx, masked: bool, saved: Optional[dict], unmasked32=None):
    """Returns the encoder input rows (bf16).  masked=True: only the visible tokens (rows [B, nv]);
    masked=False: all tokens (rows [B, n])."""
    cfg = model.cfg
    dev = A.device
    D = cfg.dim
    n_rows = geo.nv if masked else geo.n
    x0 = torch.empty((B * n_rows, D), dtype=torch.bfloat16, device=dev)
    sincos = cfg.use_sincosmod_encodings
    mods = []
    if geo.use_vision:
        ps = ops.make_patch_source([x["image"]], model.ph_img, model.pw_img, 0)
        ncols = geo.nv_img if masked else geo.n_img
        mods.append(("image", ps, 0, ncols, tabs.enc_dst_img if masked else tabs.all_dst_img,
                     tabs.enc_cls_img if masked else tabs.all_cls_img, None if masked else tabs.all_pos_img))
    if geo.nt:
        ps = ops.make_patch_source([x[f"tactile{i + 1}"] for i in range(geo.nt)], model.ph_tac, model.pw_tac, geo.n_img)
        ncols = geo.nv_tac if masked else geo.nt * geo.n_tac
        mods.append(("tactile", ps, geo.nv_img if masked else 0, ncols, tabs.enc_dst_tac if masked else tabs.all_dst_tac,
                     tabs.enc_cls_tac if masked else tabs.all_cls_tac, None if masked else tabs.all_pos_tac))
    def embed_one(name, ps, col0, ncols, dst, cls_rows, pos_rows):
        pre = f"{name}_patch_to_emb"
        a, xhat = ops.patch_layernorm(ps, B, ncols, A.f32(pre + ".0.weight"), A.f32(pre + ".0.bias"),
                                      tok_idx=tok_idx if masked else None, col0=col0, want_xhat=saved is not None)
        e = ops.gemm(a, A.bf(pre + ".1.weight"), bias=A.f32(pre + ".1.bias"), out_dtype=torch.float32)
        if masked:
            # position row of embedding row (b, jj) = unmasked[b, col0 + jj]
            pos_rows = unmasked32[:, col0:col0 + ncols].contiguous().view(-1)
        if sincos:
            add0, add0_row, add1, add1_row = A.f32("encoder_modality_embedding.weight"), cls_rows, tabs.enc_pos, pos_rows
        else:
            add0 = add0_row = None
            add1, add1_row = A.f32("encoder.pos_embedding")[0, 1:geo.n + 1], pos_rows
        _, st = ops.layernorm_fwd(e, A.f32(pre + ".2.weight"), A.f32(pre + ".2.bias"), out=x0, dst_row=dst,
                                  add0=add0, add0_row=add0_row, add1=add1, add1_row=add1_row,
                                  want_stats=saved is not None)
        if saved is not None:
            saved[name] = (a, xhat, e, st, dst, pos_rows)

    # image and tactile embeddings write disjoint rows of x0: parallel branches
    br = Branch(dev, enabled=len(mods) == 2)
    with br:
        embed_one(*mods[0])
    for m in mods[1:]:
        embed_one(*m)
    br.join()
    return x0


def _embed_bwd(model, A, G, geo, tabs, dx0, B, masked: bool, saved: dict):
    cfg = model.cfg
    n_rows = geo.nv if masked else geo.n
    # broadcast adds: modality embedding / learned positions (only reads dx0: a branch of its own, beside the
    # per-modality chains below)
    br0 = Branch(A.device, index=3)
    with br0:
        if cfg.use_sincosmod_encodings:
            if masked:
                ops.rowclass_sum(dx0, B, n_rows, slot_class=tabs.slot_class, dclass=G("encoder_modality_embedding.weight"))
            else:
                ops.rowclass_sum(dx0, B, n_rows, slot_class=tabs.tok_class, dclass=G("encoder_modality_embedding.weight"))
        else:
            gpos = G("encoder.pos_embedding")[0, 1:geo.n + 1]
            if masked:
                ops.rowclass_sum(dx0, B, n_rows, row_pos=saved["unmasked32"].view(-1), dpos=gpos)
            else:
                pos = torch.arange(geo.n, device=dx0.device, dtype=torch.int32).repeat(B)
                ops.rowclass_sum(dx0, B, n_rows, row_pos=pos, dpos=gpos)

    def embed_bwd_one(name):
        pre = f"{name}_patch_to_emb"
        a, xhat, e, st, dst, _ = saved[name]
        de = ops.layernorm_bwd(dx0, e, st, A.f32(pre + ".2.weight"), dgamma=G(pre + ".2.weight"),
                               dbeta=G(pre + ".2.bias"), src_row=dst)
        ops.colsum(de, G(pre + ".1.bias"))
        wgrad(de, a, G(pre + ".1.weight"))
        da = ops.gemm(de, A.bf_t(pre + ".1.weight"))
        ops.ln_param_grad(da, xhat, G(pre + ".0.weight"), G(pre + ".0.bias"))
        return de, da                    # kept alive until the branches have joined

    names = [nm for nm in ("image", "tactile") if nm in saved]
    br = Branch(A.device, enabled=len(names) == 2)
    with br:
        keep = [embed_bwd_one(names[0])]
    for nm in names[1:]:
        keep.append(embed_bwd_one(nm))
    br.join()
    br0.join()
    del keep


# --------------------------------------------------------------------------------------------
# masked-autoencoder forward / backward
# --------------------------------------------------------------------------------------------
def mae_forward(model, x: Dict[str, torch.Tensor], noise: torch.Tensor, geo: Geometry, training: bool,
                gflat: Optional[torch.Tensor] = None, capture: Optional[dict] = None,
                tokens_all: Optional[torch.Tensor] = None):
    """Returns (loss_acc fp32[1], ctx).  ctx holds what mae_backward needs (None if not training).
    gflat: the (zeroed) flat gradient buffer the backward pass will use; when given, the MSE kernel
    already accumulates the head bias gradients (column sums of dpred) into it.
    tokens_all: the embedded token sequence of ALL tokens [B*n, dim] (joint step: computed once for this pass and for
    the feature extractor); the masked encoder's input is then a row gather of it and the embedding's backward is left
    to the caller (mae_backward_encoder returns the gradient w.r.t. the gathered rows)."""
    cfg, A = model.cfg, model.arena
    dev = A.device
    B = noise.shape[0]
    tabs = model.tables(geo, B)
    ctx = {"geo": geo, "B": B, "x": x} if training else None
    masked, unmasked, slots, unmasked32, mrow = ops.mask_indices(noise, geo.segs, extra=True, n_masked_first=geo.nm_img)
    model.last_masked_indices, model.last_unmasked_indices = masked, unmasked
    emb_saved = {"unmasked32": unmasked32} if training else None
    ecm = cfg.early_conv_masking
    if tokens_all is not None:
        x0 = torch.empty((B * geo.nv, cfg.dim), dtype=torch.bfloat16, device=dev)
        ops.token_finish(tokens_all, B, geo.n, geo.nv, 0, x0, tok_idx=unmasked32)        # tokens[b, visible] (:256)
        if training:
            emb_saved["shared"] = True
    elif ecm:
        x0 = _embed_fwd_ecm(model, A, geo, tabs, x, B, True, emb_saved, unmasked32=unmasked32)
    else:
        x0 = _embed_fwd(model, A, geo, tabs, x, B, unmasked, True, emb_saved, unmasked32=unmasked32)
    enc_saved = [] if training else None
    xe = stack_fwd(A, model.enc_spec, x0, B, geo.nv, enc_saved, p_drop=p_drop(model.encoder.transformer))
    enc_out, st_enc = ops.layernorm_fwd(xe, A.f32("encoder.transformer.norm.weight"), A.f32("encoder.transformer.norm.bias"),
                                        want_stats=training)
    if model.has_enc_to_dec:
        d = ops.gemm(enc_out, A.bf("enc_to_dec.weight"), bias=A.f32("enc_to_dec.bias"))
    else:
        d = enc_out
    if cfg.use_sincosmod_encodings:
        z = ops.decoder_assemble_fwd(d, geo.nv, A.f32("mask_token"), slots, B, geo.n,
                                     add0=A.f32("decoder_modality_embedding.weight"), tok_class=tabs.tok_class,
                                     add1=tabs.dec_pos)
    else:
        z = ops.decoder_assemble_fwd(d, geo.nv, A.f32("mask_token"), slots, B, geo.n,
                                     add1=A.f32("decoder_pos_emb.weight")[:geo.n])
    dec_saved = [] if training else None
    xd = stack_fwd(A, model.dec_spec, z, B, geo.n, dec_saved)
    # final LayerNorm, written straight into the stacked head inputs (masked rows only; with
    # early_conv_masking the heads and the loss cover ALL tokens: pretrain_models.py:311-322)
    if ecm:
        mrow = tabs.head_row_all
    h_img, h_tac = (geo.n_img, geo.nt * geo.n_tac) if ecm else (geo.nm_img, geo.nm_tac_total)
    gathered, st_dec = ops.layernorm_fwd(xd, A.f32("decoder.norm.weight"), A.f32("decoder.norm.bias"),
                                         out_rows=B * (h_img + h_tac), dst_row=mrow, want_stats=training)
    loss_acc = torch.zeros(1, dtype=torch.float32, device=dev)
    heads = []
    G = GradView(A, gflat) if (training and gflat is not None) else None
    r_img = B * h_img

    def head(name, g_in, maps, ph, pw, tok_base, h_cols, weight, col0, row0, cap_key, ws_slot):
        pred = ops.gemm(g_in, A.bf(name + ".weight"), bias=A.f32(name + ".bias"), out_dtype=torch.float32)
        ps = ops.make_patch_source(maps, ph, pw, tok_base)
        dpred = ops.mse_loss(ps, B, h_cols, pred, weight / pred.numel(), loss_acc, tok_idx=None if ecm else masked, col0=col0,
                             dpred_colsum=G(name + ".bias") if G is not None and pred.shape[1] <= 1024 else None,
                             ws_slot=ws_slot)
        heads.append((name, g_in, dpred, row0))
        if capture is not None:
            capture[cap_key] = pred

    # the two heads (GEMM + masked-patch MSE each) are independent: parallel branches
    br = Branch(dev, enabled=bool(geo.nt) and geo.use_vision)
    if geo.nt:
        with br:
            head("to_tactiles", gathered[r_img:], [x[f"tactile{i + 1}"] for i in range(geo.nt)], model.ph_tac, model.pw_tac,
                 geo.n_img, h_tac, 10.0, geo.nm_img, r_img, "pred_tactile", 1)
    if geo.use_vision:
        head("to_pixels", gathered[:r_img], [x["image"]], model.ph_img, model.pw_img, 0, h_img, 1.0, 0, 0, "pred_image", 0)
    br.join()
    if training:
        ctx.update(tabs=tabs, slots=slots, mrow=mrow, emb=emb_saved, enc=enc_saved, xe=xe, st_enc=st_enc,
                   enc_out=enc_out, dec=dec_saved, xd=xd, st_dec=st_dec, heads=heads, n_gathered=gathered.shape[0],
                   gflat_fwd=gflat)
    return loss_acc, ctx


def mae_backward_decoder(model, ctx, gflat: torch.Tensor):
    """Heads + decoder part of the backward (its gradients are final first: SURVEY.md §8e)."""
    cfg, A = model.cfg, model.arena
    G = GradView(A, gflat)
    geo, B, tabs = ctx["geo"], ctx["B"], ctx["tabs"]
    Dd = cfg.decoder_dim
    dgath = torch.empty((ctx["n_gathered"], Dd), dtype=torch.bfloat16, device=A.device)
    bias_done = ctx.get("gflat_fwd") is gflat and gflat is not None   # fused into the MSE kernel
    def head_bwd(name, g_in, dpred, row0):
        if not (bias_done and dpred.shape[1] <= 1024):
            ops.colsum(dpred, G(name + ".bias"))
        wgrad(dpred, g_in, G(name + ".weight"))
        ops.gemm(dpred, A.bf_t(name + ".weight"), out=dgath[row0:row0 + g_in.shape[0]])

    hs = ctx["heads"]
    br = Branch(A.device, enabled=len(hs) == 2)
    with br:
        head_bwd(*hs[0])
    for h_ in hs[1:]:
        head_bwd(*h_)
    br.join()
    dxd = ops.layernorm_bwd(dgath, ctx["xd"], ctx["st_dec"], A.f32("decoder.norm.weight"),
                            dgamma=G("decoder.norm.weight"), dbeta=G("decoder.norm.bias"), src_row=ctx["mrow"],
                            dx_colsum=G(last_ff_bias(model.dec_spec)))
    dz = stack_bwd(A, G, model.dec_spec, dxd, B, geo.n, ctx["dec"])
    if cfg.use_sincosmod_encodings:
        dd = ops.decoder_assemble_bwd(dz, ctx["slots"], B, geo.n, geo.nv, dmask_token=G("mask_token"),
                                      dadd0=G("decoder_modality_embedding.weight"), tok_class=tabs.tok_class)
    else:
        dd = ops.decoder_assemble_bwd(dz, ctx["slots"], B, geo.n, geo.nv, dmask_token=G("mask_token"),
                                      dadd1=G("decoder_pos_emb.weight")[:geo.n])
    ctx["dd"] = dd
    if model.has_enc_to_dec:
        # enc_to_dec's parameter gradients belong to the FIRST all-reduce bucket (dp.DECODER_SIDE_PREFIXES), so they
        # must be final when this phase ends; only the dgrad through it is left to the encoder phase
        ops.colsum(dd, G("enc_to_dec.bias"))
        wgrad(dd, ctx["enc_out"], G("enc_to_dec.weight"))


def mae_backward_encoder_stack(model, ctx, gflat: torch.Tensor):
    """Encoder transformer part of the backward; returns the gradient w.r.t. the encoder input rows."""
    A = model.arena
    G = GradView(A, gflat)
    geo, B = ctx["geo"], ctx["B"]
    dd = ctx["dd"]
    if model.has_enc_to_dec:
        denc = ops.gemm(dd, A.bf_t("enc_to_dec.weight"))
    else:
        denc = dd
    dxe = ops.layernorm_bwd(denc, ctx["xe"], ctx["st_enc"], A.f32("encoder.transformer.norm.weight"),
                            dgamma=G("encoder.transformer.norm.weight"), dbeta=G("encoder.transformer.norm.bias"),
                            dx_colsum=stack_dx_colsum(G, model.enc_spec, ctx["enc"]))
    return stack_bwd(A, G, model.enc_spec, dxe, B, geo.nv, ctx["enc"])


def mae_backward_embed(model, ctx, gflat: torch.Tensor, dx0: torch.Tensor):
    """Token-embedding part of the backward (patch embeddings / conv stems, modality and position tables)."""
    cfg, A = model.cfg, model.arena
    G = GradView(A, gflat)
    geo, B, tabs = ctx["geo"], ctx["B"], ctx["tabs"]
    if cfg.early_conv_masking:
        _embed_bwd_ecm(model, A, G, geo, tabs, dx0, B, True, ctx["emb"], slots=ctx["slots"])
    else:
        _embed_bwd(model, A, G, geo, tabs, dx0, B, True, ctx["emb"])


def mae_backward_encoder(model, ctx, gflat: torch.Tensor):
    dx0 = mae_backward_encoder_stack(model, ctx, gflat)
    if ctx["emb"].get("shared"):
        return dx0                       # joint step: the caller adds it into the full-sequence gradient
    mae_backward_embed(model, ctx, gflat, dx0)
    return None


# --------------------------------------------------------------------------------------------
# no-mask encoder pass (get_embeddings)
# --------------------------------------------------------------------------------------------
def embeddings_forward(model, x, geo: Geometry, B: int, training: bool):
    A = model.arena
    tabs = model.tables(geo, B)
    emb_saved = {} if training else None
    if model.cfg.early_conv_masking:
        x0 = _embed_fwd_ecm(model, A, geo, tabs, x, B, False, emb_saved)
    else:
        x0 = _embed_fwd(model, A, geo, tabs, x, B, None, False, emb_saved)
    enc_saved = [] if training else None
    xe = stack_fwd(A, model.enc_spec, x0, B, geo.n, enc_saved, p_drop=p_drop(model.encoder.transformer))
    out, st = ops.layernorm_fwd(xe, A.f32("encoder.transformer.norm.weight"), A.f32("encoder.transformer.norm.bias"),
                                want_stats=training)
    ctx = dict(geo=geo, B=B, tabs=tabs, emb=emb_saved, enc=enc_saved, xe=xe, st=st, tokens_all=x0) if training else None
    return out, ctx


def embeddings_backward(model, ctx, dout: torch.Tensor, gflat: torch.Tensor, extra_token_grad=None):
    """extra_token_grad: optional (dx_rows bf16 [B*k, dim], tok_idx int32 [B, k]) added into the gradient of the embedded
    token sequence before the embedding's backward (the masked-autoencoder branch of the joint step)."""
    A = model.arena
    G = GradView(A, gflat)
    geo, B, tabs = ctx["geo"], ctx["B"], ctx["tabs"]
    dxe = ops.layernorm_bwd(dout, ctx["xe"], ctx["st"], A.f32("encoder.transformer.norm.weight"),
                            dgamma=G("encoder.transformer.norm.weight"), dbeta=G("encoder.transformer.norm.bias"),
                            dx_colsum=stack_dx_colsum(G, model.enc_spec, ctx["enc"]))
    dx0 = stack_bwd(A, G, model.enc_spec, dxe, B, geo.n, ctx["enc"])
    if extra_token_grad is not None:
        ops.row_scatter_add(extra_token_grad[0], extra_token_grad[1], B, geo.n, dx0)
    if model.cfg.early_conv_masking:
        _embed_bwd_ecm(model, A, G, geo, tabs, dx0, B, False, ctx["emb"])
    else:
        _embed_bwd(model, A, G, geo, tabs, dx0, B, False, ctx["emb"])
