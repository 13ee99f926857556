"""Python wrappers of the individual C-ABI kernels (unit-test and composition surface).

Every function takes CUDA torch tensors, passes raw pointers + the current stream to the
C-ABI and returns torch tensors.  torch is only the allocator / stream provider here.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Optional

import torch

from . import _lib
from ._lib import GemmArgs, check, current_stream, ptr

GELU_FWD = 1
GELU_BWD = 2
RELU = 3


class Dropout(NamedTuple):
    """One dropout site of a training pass: key int64 [1] on the device, site = (layer << 2) | s (s = 0 attention
    probabilities, 1 attention output, 2 after GELU, 3 feed-forward output), p in [0, 1).  The mask is the
    counter-based one of csrc/dropout.cuh (include/m3l_b200.h)."""
    key: torch.Tensor
    site: int
    p: float


def _drop_args(d: Optional[Dropout]):
    if d is None:
        return C.c_void_p(0), 0, C.c_float(0.0)
    assert d.key.dtype == torch.int64 and d.key.is_cuda and d.key.numel() >= 1
    return ptr(d.key), int(d.site), C.c_float(d.p)


_WS = {}
_WS_BYTES = 1 << 20


def workspace(device, slot: int = 0):
    """Zero-initialised reduction scratch, one per (device, slot) (kernels restore the leading counter to 0).
    Kernels that may run concurrently on two streams (the two reconstruction heads) use different slots."""
    key = (device.type, device.index, slot)
    ws = _WS.get(key)
    if ws is None:
        ws = torch.zeros(_WS_BYTES, dtype=torch.uint8, device=device)
        _WS[key] = ws
    return ws


def _req_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.M3LError("m3l_b200 ops need CUDA tensors (there is no CPU fallback)")


def gemm(a: torch.Tensor, b: torch.Tensor, *, mn_major: bool = False, out: Optional[torch.Tensor] = None,
         out_dtype: torch.dtype = torch.bfloat16, accumulate: bool = False, splits: int = 1, bn: int = 0,
         bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None, act: int = 0,
         aux_out: Optional[torch.Tensor] = None, aux_in: Optional[torch.Tensor] = None,
         alpha: float = 1.0, colsum_out: Optional[torch.Tensor] = None,
         dot_side: Optional[torch.Tensor] = None, dot_out: Optional[torch.Tensor] = None,
         out2: Optional[torch.Tensor] = None, ln_bwd: Optional[dict] = None,
         dropout: Optional[Dropout] = None) -> torch.Tensor:
    """out[m, n] = epilogue(alpha * sum_k A[m, k] B[n, k]).

    mn_major=False: a is [M, K], b is [N, K] (nn.Linear forward: x @ W.T).
    mn_major=True : a is [K, M], b is [K, N] (wgrad: a.T @ b), optionally split-K + accumulate.
    dropout: with act=GELU_FWD, out = Z o GELU and aux_out = Z o GELU'; with a residual (act 0),
    out = residual + Z o (acc + bias).  Other epilogues reject it.
    """
    _req_cuda(a, b, out, bias, residual, aux_out, aux_in)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    assert a.dim() == 2 and b.dim() == 2 and a.stride(1) == 1 and b.stride(1) == 1
    if mn_major:
        K, M = a.shape
        K2, N = b.shape
    else:
        M, K = a.shape
        N, K2 = b.shape
    assert K == K2, (a.shape, b.shape)
    if out is None:
        dt = torch.float32 if accumulate else out_dtype
        out = (torch.zeros if accumulate else torch.empty)((M, N), dtype=dt, device=a.device)
    assert out.stride(1) == 1
    if accumulate:
        assert out.dtype == torch.float32
        out_mode = 2
    else:
        out_mode = 0 if out.dtype == torch.bfloat16 else 1
    args = GemmArgs()
    args.a, args.b = ptr(a), ptr(b)
    args.lda, args.ldb = a.stride(0), b.stride(0)
    args.a_mn_major = args.b_mn_major = 1 if mn_major else 0
    args.m, args.n, args.k = M, N, K
    args.splits, args.bn = splits, bn
    args.out, args.ldo, args.out_mode = ptr(out), out.stride(0), out_mode
    args.bias = ptr(bias)
    args.residual, args.ldr = ptr(residual), (residual.stride(0) if residual is not None else 0)
    args.act = act
    args.aux_out, args.aux_in = ptr(aux_out), ptr(aux_in)
    aux = aux_out if aux_out is not None else aux_in
    args.ld_aux = aux.stride(0) if aux is not None else 0
    args.alpha = alpha
    args.colsum_out = ptr(colsum_out)
    if out2 is not None:
        assert out2.dtype == torch.bfloat16 and out2.shape == out.shape and out2.stride() == out.stride()
        args.out2 = ptr(out2)
    if dot_side is not None:
        assert dot_side.dtype == torch.bfloat16 and dot_side.stride(1) == 1 and dot_side.shape == (M, N)
        assert dot_out is not None and dot_out.dtype == torch.float32 and dot_out.is_contiguous() and dot_out.shape == (M, N // 64)
        args.dot_side, args.ld_dot, args.dot_out = ptr(dot_side), dot_side.stride(0), ptr(dot_out)
    if ln_bwd is not None:
        # fused LayerNorm backward epilogue: out = dLN(a @ b.T; x, stats, gamma) (+ skip); dgamma / dbeta / dxcol accumulated
        x, st, gm = ln_bwd["x"], ln_bwd["stats"], ln_bwd["gamma"]
        assert N == 256 and out.dtype == torch.bfloat16 and x.shape == (M, N) and x.dtype == torch.bfloat16 and x.is_contiguous()
        assert st.shape == (M, 2) and st.dtype == torch.float32 and gm.dtype == torch.float32 and gm.numel() == N
        sk = ln_bwd.get("skip")
        assert sk is None or (sk.shape == (M, N) and sk.dtype == torch.bfloat16 and sk.is_contiguous())
        args.ln_x, args.ln_stats, args.ln_gamma, args.ln_skip = ptr(x), ptr(st), ptr(gm), ptr(sk)
        args.ln_dgamma, args.ln_dbeta, args.ln_dxcol = ptr(ln_bwd["dgamma"]), ptr(ln_bwd["dbeta"]), ptr(ln_bwd.get("dx_colsum"))
    if dropout is not None:
        args.drop_key, args.drop_site, args.drop_p = _drop_args(dropout)
    check(_lib.load().m3l_gemm_bf16(C.byref(args), current_stream()), "m3l_gemm_bf16")
    return out


def ln_mlp_supported(dim: int, hidden: int) -> bool:
    """Shapes the fused feed-forward block kernel is built for (csrc/rowblock.cu)."""
    return dim == 256 and hidden % 128 == 0 and 128 <= hidden <= 1024


def ln_mlp_fwd(x, gamma, beta, w1, b1, w2, b2, *, save: bool = False, eps: float = 1e-5, out=None,
               out_has_x: bool = False):
    """out = x + W2 GELU(W1 LayerNorm(x) + b1) + b2 in one kernel (x bf16 [M, 256]; w1 [hidden, 256], w2 [256, hidden] bf16).
    out=x updates the residual stream in place; out_has_x=True says `out` already holds a copy of x (gemm(out2=...)): in
    both cases the block output is reduce-added to out and x is read once.
    save=True additionally returns what the backward pass reads: (out, stats, xn, h, gelu_grad)."""
    _req_cuda(x, gamma, beta, w1, b1, w2, b2, out)
    M, D = x.shape
    hidden = w1.shape[0]
    assert x.dtype == torch.bfloat16 and x.is_contiguous() and w1.is_contiguous() and w2.is_contiguous()
    assert w1.shape == (hidden, D) and w2.shape == (D, hidden) and w1.dtype == torch.bfloat16 and w2.dtype == torch.bfloat16
    if out is None:
        assert not out_has_x
        if save:                      # the training outputs go with the accumulate-into-out mode of the kernel
            out, out_has_x = x.clone(), True
        else:
            out = torch.empty_like(x)
    assert out.shape == x.shape and out.dtype == torch.bfloat16 and out.is_contiguous()
    a = _lib.LnMlpArgs()
    a.x, a.rows, a.dim, a.hidden = ptr(x), M, D, hidden
    a.gamma, a.beta, a.eps = ptr(gamma), ptr(beta), eps
    a.w1, a.b1, a.w2, a.b2 = ptr(w1), ptr(b1), ptr(w2), ptr(b2)
    a.out, a.out_has_x = ptr(out), int(out_has_x)
    stats = xn = h = gp = None
    if save:
        stats = torch.empty((M, 2), dtype=torch.float32, device=x.device)
        xn = torch.empty_like(x)
        h = torch.empty((M, hidden), dtype=torch.bfloat16, device=x.device)
        gp = torch.empty_like(h)
        a.stats, a.xn_out, a.h_out, a.gp_out = ptr(stats), ptr(xn), ptr(h), ptr(gp)
    check(_lib.load().m3l_ln_mlp_fwd(C.byref(a), current_stream()), "m3l_ln_mlp_fwd")
    if save:
        return out, stats, xn, h, gp
    return out


# ------------------------------------------------------------------------------------------
# mask sampling / patch sources
# ------------------------------------------------------------------------------------------
def make_segments(segs):
    """segs: list of (offset, length, n_masked)."""
    s = _lib.MaskSegments()
    s.count = len(segs)
    for i, (o, l, m) in enumerate(segs):
        s.offset[i], s.length[i], s.n_masked[i] = o, l, m
    return s


def mask_indices(noise: torch.Tensor, segs, want_slots: bool = True, extra: bool = False, n_masked_first: int = 0):
    """noise fp32 [B, n_total] -> (masked int64 [B, nm], unmasked int64 [B, nu], slot_of_token int32 [B, n]).
    extra=True additionally returns (unmasked int32, masked_row_of_token int32 [B, n])."""
    _req_cuda(noise)
    assert noise.dtype == torch.float32 and noise.is_contiguous()
    B, n = noise.shape
    nm = sum(m for _, _, m in segs)
    nu = sum(l - m for _, l, m in segs)
    masked = torch.empty((B, nm), dtype=torch.int64, device=noise.device)
    unmasked = torch.empty((B, nu), dtype=torch.int64, device=noise.device)
    slots = torch.empty((B, n), dtype=torch.int32, device=noise.device) if want_slots else None
    cs = make_segments(segs)
    u32 = torch.empty((B, nu), dtype=torch.int32, device=noise.device) if extra else None
    mrow = torch.empty((B, n), dtype=torch.int32, device=noise.device) if extra else None
    check(_lib.load().m3l_mask_indices(ptr(noise), B, n, C.byref(cs), ptr(masked), ptr(unmasked), ptr(slots),
                                       ptr(u32), ptr(mrow), n_masked_first, current_stream()), "m3l_mask_indices")
    if extra:
        return masked, unmasked, slots, u32, mrow
    return masked, unmasked, slots


def make_patch_source(maps, patch_h: int, patch_w: int, token_base: int):
    """maps: list of fp32 NCHW tensors of one modality (same shape), or of data.RawMap views into raw observation
    tensors (vt_load fused into the patch loads: `layout 1` of m3l_patch_source)."""
    from .data import RawMap
    ps = _lib.PatchSource()
    assert 1 <= len(maps) <= 4
    if isinstance(maps[0], RawMap):
        m0 = maps[0]
        for i, m in enumerate(maps):
            assert isinstance(m, RawMap) and m.is_cuda and m.shape == m0.shape and m.t.dtype == m0.t.dtype
            assert (m.sb, m.cg, m.sf, m.sch, m.sy, m.sx, m.lo, m.span) == (m0.sb, m0.cg, m0.sf, m0.sch, m0.sy, m0.sx, m0.lo, m0.span)
            ps.src[i] = m.data_ptr()
        _, ps.channels, ps.height, ps.width = m0.shape
        ps.layout, ps.dtype = 1, (1 if m0.t.dtype == torch.uint8 else 0)
        ps.stride_b, ps.chan_group = m0.sb, m0.cg
        ps.stride_f, ps.stride_ch, ps.stride_y, ps.stride_x = m0.sf, m0.sch, m0.sy, m0.sx
        ps.norm_lo, ps.norm_span = m0.lo, m0.span
    else:
        for i, m in enumerate(maps):
            assert m.dtype == torch.float32 and m.is_contiguous() and m.is_cuda and m.shape == maps[0].shape
            ps.src[i] = m.data_ptr()
        _, ps.channels, ps.height, ps.width = maps[0].shape
    ps.patch_h, ps.patch_w, ps.token_base = patch_h, patch_w, token_base
    ps._keepalive = maps
    return ps


def vt_load_map(raw, out=None) -> torch.Tensor:
    """data.RawMap -> fp32 [B, C, H, W] contiguous (utils/pretrain_utils.py:7-57 as one kernel)."""
    ps = make_patch_source([raw], 1, 1, 0)
    B = raw.shape[0]
    if out is None:
        out = torch.empty(raw.shape, dtype=torch.float32, device=raw.device)
    assert out.shape == tuple(raw.shape) and out.dtype == torch.float32 and out.is_contiguous()
    check(_lib.load().m3l_vt_load(C.byref(ps), B, 0, ptr(out), current_stream()), "m3l_vt_load")
    return out


def patch_layernorm(ps, batch: int, ncols: int, gamma, beta, tok_idx=None, col0: int = 0, want_xhat=True,
                    eps: float = 1e-5):
    P = ps.patch_h * ps.patch_w * ps.channels
    dev = gamma.device
    out = torch.empty((batch * ncols, P), dtype=torch.bfloat16, device=dev)
    xhat = torch.empty_like(out) if want_xhat else None
    idx_ld = tok_idx.stride(0) if tok_idx is not None else 0
    check(_lib.load().m3l_patch_layernorm(C.byref(ps), batch, ptr(tok_idx), idx_ld, col0, ncols, ptr(gamma),
                                          ptr(beta), C.c_float(eps), ptr(out), ptr(xhat), current_stream()),
          "m3l_patch_layernorm")
    return out, xhat


def patchify(ps, batch: int, ncols: int, *, ld: int = 0, tok_idx=None, col0: int = 0):
    """Patch rows bf16 [batch*ncols, ld] in (p1, p2, c) order, zero-padded to the row pitch ld (default: P rounded up to 8)."""
    P = ps.patch_h * ps.patch_w * ps.channels
    ld = ld or (P + 7) // 8 * 8
    dev = ps._keepalive[0].device
    out = torch.empty((batch * ncols, ld), dtype=torch.bfloat16, device=dev)
    idx_ld = tok_idx.stride(0) if tok_idx is not None else 0
    check(_lib.load().m3l_patchify(C.byref(ps), batch, ptr(tok_idx), idx_ld, col0, ncols, ptr(out), ld, current_stream()),
          "m3l_patchify")
    return out


def layernorm_fwd(x, gamma, beta, *, out=None, out_rows=None, stats=None, want_stats=True, dst_row=None,
                  add0=None, add0_row=None, add1=None, add1_row=None, eps: float = 1e-5):
    _req_cuda(x, gamma, beta)
    M, D = x.shape
    assert x.is_contiguous() and x.dtype in (torch.bfloat16, torch.float32)
    if out is None:
        out = torch.empty((out_rows if out_rows is not None else M, D), dtype=torch.bfloat16, device=x.device)
    if stats is None and want_stats:
        stats = torch.empty((M, 2), dtype=torch.float32, device=x.device)
    check(_lib.load().m3l_layernorm_fwd(ptr(x), int(x.dtype == torch.float32), M, D, ptr(gamma), ptr(beta),
                                        C.c_float(eps), ptr(out), ptr(stats), ptr(dst_row), ptr(add0),
                                        ptr(add0_row), ptr(add1), ptr(add1_row), current_stream()),
          "m3l_layernorm_fwd")
    return out, stats


def layernorm_bwd(dy, x, stats, gamma, *, dgamma=None, dbeta=None, skip=None, src_row=None, dx=None,
                  dx_dtype=torch.bfloat16, dx_colsum=None):
    _req_cuda(dy, x, stats, gamma)
    M, D = x.shape
    if dx is None:
        dx = torch.empty((M, D), dtype=dx_dtype, device=x.device)
    check(_lib.load().m3l_layernorm_bwd(ptr(dy), ptr(src_row), ptr(x), int(x.dtype == torch.float32), ptr(stats),
                                        M, D, ptr(gamma), ptr(skip), ptr(dx), int(dx.dtype == torch.float32),
                                        ptr(dgamma), ptr(dbeta), ptr(dx_colsum), current_stream()),
          "m3l_layernorm_bwd")
    return dx


def decoder_assemble_fwd(d, n_visible, mask_token, slots, batch, n_tokens, *, add0=None, tok_class=None,
                         add1=None, out=None):
    D = d.shape[-1]
    if out is None:
        out = torch.empty((batch * n_tokens, D), dtype=torch.bfloat16, device=d.device)
    check(_lib.load().m3l_decoder_assemble_fwd(ptr(d), n_visible, ptr(mask_token), ptr(slots), batch, n_tokens, D,
                                               ptr(add0), ptr(tok_class), ptr(add1), ptr(out), current_stream()),
          "m3l_decoder_assemble_fwd")
    return out


def decoder_assemble_bwd(dz, slots, batch, n_tokens, n_visible, *, dmask_token=None, dadd0=None, tok_class=None,
                         dadd1=None, out=None):
    D = dz.shape[-1]
    if out is None:
        out = torch.empty((batch * n_visible, D), dtype=torch.bfloat16, device=dz.device)
    n_classes = dadd0.shape[0] if dadd0 is not None else 0
    check(_lib.load().m3l_decoder_assemble_bwd(ptr(dz), ptr(slots), batch, n_tokens, D, n_visible, ptr(out),
                                               ptr(dmask_token), ptr(dadd0), ptr(tok_class), n_classes, ptr(dadd1),
                                               current_stream()), "m3l_decoder_assemble_bwd")
    return out


def rowclass_sum(dx, batch, n_visible, *, slot_class=None, dclass=None, row_pos=None, dpos=None):
    check(_lib.load().m3l_rowclass_sum(ptr(dx), batch, n_visible, dx.shape[-1], ptr(slot_class), ptr(dclass),
                                       ptr(row_pos), ptr(dpos), current_stream()), "m3l_rowclass_sum")


def mse_loss(ps, batch, ncols, pred, weight, loss_acc, *, tok_idx=None, col0=0, dpred=None, dpred_colsum=None,
             ws_slot: int = 0):
    assert pred.dtype == torch.float32 and pred.is_contiguous()
    if dpred is None:
        dpred = torch.empty(pred.shape, dtype=torch.bfloat16, device=pred.device)
    idx_ld = tok_idx.stride(0) if tok_idx is not None else 0
    check(_lib.load().m3l_mse_loss(C.byref(ps), batch, ptr(tok_idx), idx_ld, col0, ncols, ptr(pred),
                                   C.c_float(weight), ptr(dpred), ptr(loss_acc), ptr(dpred_colsum),
                                   ptr(workspace(pred.device, ws_slot)),
                                   C.c_size_t(_WS_BYTES), current_stream()), "m3l_mse_loss")
    return dpred


def colsum(x, out):
    assert x.dtype == torch.bfloat16 and x.stride(1) == 1 and out.dtype == torch.float32
    check(_lib.load().m3l_colsum(ptr(x), x.shape[0], x.shape[1], x.stride(0), ptr(out), current_stream()),
          "m3l_colsum")
    return out


def ln_param_grad(da, xhat, dgamma, dbeta):
    check(_lib.load().m3l_ln_param_grad(ptr(da), ptr(xhat), da.shape[0], da.shape[1], ptr(dgamma), ptr(dbeta),
                                        current_stream()), "m3l_ln_param_grad")


# ------------------------------------------------------------------------------------------
# EarlyCNN conv stem (im2col + GEMM)
# ------------------------------------------------------------------------------------------
def conv_out_size(size, k, stride, pad):
    return (size + 2 * pad - k) // stride + 1


def im2col(x, batch, channels, height, width, k, stride, pad, nhwc_bf16, out=None):
    """x: fp32 NCHW maps (nhwc_bf16=False) or bf16 [B*H*W, C] (True) -> bf16 [B*Ho*Wo, C*k*k]."""
    _req_cuda(x)
    assert x.is_contiguous() and x.dtype == (torch.bfloat16 if nhwc_bf16 else torch.float32)
    ho, wo = conv_out_size(height, k, stride, pad), conv_out_size(width, k, stride, pad)
    col = out if out is not None else torch.empty((batch * ho * wo, channels * k * k), dtype=torch.bfloat16, device=x.device)
    assert col.shape == (batch * ho * wo, channels * k * k) and col.is_contiguous() and col.dtype == torch.bfloat16
    check(_lib.load().m3l_im2col(ptr(x), 1 if nhwc_bf16 else 0, batch, channels, height, width, k, stride, pad, ptr(col),
                                 current_stream()), "m3l_im2col")
    return col


def col2im_relu(dcol, batch, channels, height, width, k, stride, pad, relu_out=None):
    """dcol bf16 [B*Ho*Wo, C*k*k] -> dx bf16 [B*H*W, C] (x [relu_out > 0] when given)."""
    _req_cuda(dcol, relu_out)
    assert dcol.dtype == torch.bfloat16 and dcol.is_contiguous()
    dx = torch.empty((batch * height * width, channels), dtype=torch.bfloat16, device=dcol.device)
    check(_lib.load().m3l_col2im_relu(ptr(dcol), batch, channels, height, width, k, stride, pad, ptr(relu_out), ptr(dx),
                                      current_stream()), "m3l_col2im_relu")
    return dx


def token_finish(x, batch, n_per, ncols, tok_base, out, *, tok_idx=None, col0=0, add0=None, tok_class=None, add1=None,
                 dst_row=None):
    _req_cuda(x, out)
    assert x.dtype == torch.bfloat16 and x.is_contiguous() and out.dtype == torch.bfloat16
    idx_ld = tok_idx.stride(0) if tok_idx is not None else 0
    assert tok_idx is None or tok_idx.dtype == torch.int32
    check(_lib.load().m3l_token_finish(ptr(x), batch, n_per, ptr(tok_idx), idx_ld, col0, ncols, tok_base, ptr(add0),
                                       ptr(tok_class), ptr(add1), ptr(dst_row), ptr(out), x.shape[1], current_stream()),
          "m3l_token_finish")
    return out


def token_finish_bwd(dx0, batch, rows_per_sample, n_total, tok_base, n_mod, n_per, *, slot_of_token=None):
    _req_cuda(dx0)
    assert dx0.dtype == torch.bfloat16 and dx0.is_contiguous()
    dtok = torch.empty((batch * n_mod, dx0.shape[1]), dtype=torch.bfloat16, device=dx0.device)
    check(_lib.load().m3l_token_finish_bwd(ptr(dx0), batch, rows_per_sample, n_total, ptr(slot_of_token), tok_base, n_mod,
                                           n_per, dx0.shape[1], ptr(dtok), current_stream()), "m3l_token_finish_bwd")
    return dtok


def row_scatter_add(src, tok_idx, batch, n_total, dst):
    """dst[b*n_total + tok_idx[b, j]] += src[b*ncols + j]  (bf16 rows; tok_idx int32 [batch, ncols], distinct per sample)."""
    _req_cuda(src, tok_idx, dst)
    assert src.dtype == torch.bfloat16 and dst.dtype == torch.bfloat16 and src.is_contiguous() and dst.is_contiguous()
    assert tok_idx.dtype == torch.int32 and tok_idx.shape[0] == batch and src.shape[0] == batch * tok_idx.shape[1]
    check(_lib.load().m3l_row_scatter_add(ptr(src), batch, tok_idx.shape[1], ptr(tok_idx), tok_idx.stride(0), n_total,
                                          src.shape[1], ptr(dst), current_stream()), "m3l_row_scatter_add")
    return dst


def token_mean_fwd(x, batch, n_tokens):
    """x bf16 [batch*n_tokens, dim] -> fp32 [batch, dim] (mean over the tokens of each sample)."""
    _req_cuda(x)
    assert x.dtype == torch.bfloat16 and x.is_contiguous() and x.shape[0] == batch * n_tokens
    out = torch.empty((batch, x.shape[1]), dtype=torch.float32, device=x.device)
    check(_lib.load().m3l_token_mean_fwd(ptr(x), batch, n_tokens, x.shape[1], ptr(out), current_stream()),
          "m3l_token_mean_fwd")
    return out


def token_mean_bwd(dout, batch, n_tokens):
    """dout fp32 [batch, dim] -> dx bf16 [batch*n_tokens, dim]."""
    _req_cuda(dout)
    assert dout.dtype == torch.float32 and dout.is_contiguous() and dout.shape[0] == batch
    dx = torch.empty((batch * n_tokens, dout.shape[1]), dtype=torch.bfloat16, device=dout.device)
    check(_lib.load().m3l_token_mean_bwd(ptr(dout), batch, n_tokens, dout.shape[1], ptr(dx), current_stream()),
          "m3l_token_mean_bwd")
    return dx


# ------------------------------------------------------------------------------------------
# attention
# ------------------------------------------------------------------------------------------
def attention_fwd(qkv, batch, n, heads, dim_head, scale, *, out=None, lse=None):
    _req_cuda(qkv)
    inner = heads * dim_head
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous() and qkv.shape == (batch * n, 3 * inner)
    if out is None:
        out = torch.empty((batch * n, inner), dtype=torch.bfloat16, device=qkv.device)
    if lse is None:
        lse = torch.empty((batch, heads, n), dtype=torch.float32, device=qkv.device)
    check(_lib.load().m3l_attention_fwd(ptr(qkv), batch, n, heads, dim_head, C.c_float(scale), ptr(out), ptr(lse),
                                        current_stream()), "m3l_attention_fwd")
    return out, lse


def attention_bwd(qkv, out, dout, lse, batch, n, heads, dim_head, scale, *, dqkv=None, delta=None):
    """delta: optional fp32 [batch*n, heads] = rowsum(dout * out) per head (gemm(dot_side=, dot_out=))."""
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    assert dout.is_contiguous() and out.is_contiguous()
    assert delta is None or (delta.dtype == torch.float32 and delta.is_contiguous() and delta.shape == (batch * n, heads))
    check(_lib.load().m3l_attention_bwd(ptr(qkv), ptr(out), ptr(dout), ptr(lse), ptr(delta), batch, n, heads, dim_head,
                                        C.c_float(scale), ptr(dqkv), current_stream()), "m3l_attention_bwd")
    return dqkv


def attention_long_fwd(qkv, batch, n, heads, dim_head, scale, *, out=None, lse=None):
    """attention_fwd for any n >= 1 (csrc/attention_long.cu: 128-key tiles, online softmax); same outputs."""
    _req_cuda(qkv)
    inner = heads * dim_head
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous() and qkv.shape == (batch * n, 3 * inner)
    if out is None:
        out = torch.empty((batch * n, inner), dtype=torch.bfloat16, device=qkv.device)
    if lse is None:
        lse = torch.empty((batch, heads, n), dtype=torch.float32, device=qkv.device)
    check(_lib.load().m3l_attention_long_fwd(ptr(qkv), batch, n, heads, dim_head, C.c_float(scale), ptr(out), ptr(lse),
                                             current_stream()), "m3l_attention_long_fwd")
    return out, lse


def attention_long_bwd(qkv, out, dout, lse, batch, n, heads, dim_head, scale, *, dqkv=None, delta=None):
    """attention_bwd for any n >= 1 (two deterministic kernels: dK / dV per key tile, dQ per query tile)."""
    _req_cuda(qkv, out, dout, lse, dqkv, delta)
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    assert dout.is_contiguous() and out.is_contiguous()
    assert delta is None or (delta.dtype == torch.float32 and delta.is_contiguous() and delta.shape == (batch * n, heads))
    check(_lib.load().m3l_attention_long_bwd(ptr(qkv), ptr(out), ptr(dout), ptr(lse), ptr(delta), batch, n, heads,
                                             dim_head, C.c_float(scale), ptr(dqkv), current_stream()),
          "m3l_attention_long_bwd")
    return dqkv


def attention_dh_fwd(qkv, batch, n, heads, dim_head, scale, *, out=None, lse=None):
    """attention_long_fwd for 32- and 128-wide heads (csrc/attention_dh.cu), any n >= 1; same outputs."""
    _req_cuda(qkv)
    inner = heads * dim_head
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous() and qkv.shape == (batch * n, 3 * inner)
    if out is None:
        out = torch.empty((batch * n, inner), dtype=torch.bfloat16, device=qkv.device)
    if lse is None:
        lse = torch.empty((batch, heads, n), dtype=torch.float32, device=qkv.device)
    check(_lib.load().m3l_attention_dh_fwd(ptr(qkv), batch, n, heads, dim_head, C.c_float(scale), ptr(out), ptr(lse),
                                           current_stream()), "m3l_attention_dh_fwd")
    return out, lse


def attention_dh_bwd(qkv, out, dout, lse, batch, n, heads, dim_head, scale, *, dqkv=None, delta=None):
    """attention_long_bwd for 32- and 128-wide heads (the same two deterministic kernels)."""
    _req_cuda(qkv, out, dout, lse, dqkv, delta)
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    assert dout.is_contiguous() and out.is_contiguous()
    assert delta is None or (delta.dtype == torch.float32 and delta.is_contiguous() and delta.shape == (batch * n, heads))
    check(_lib.load().m3l_attention_dh_bwd(ptr(qkv), ptr(out), ptr(dout), ptr(lse), ptr(delta), batch, n, heads,
                                           dim_head, C.c_float(scale), ptr(dqkv), current_stream()),
          "m3l_attention_dh_bwd")
    return dqkv


def attention_dropout_fwd(qkv, batch, n, heads, dim_head, scale, dropout: Dropout, *, out=None, lse=None):
    """attention_long_fwd / attention_dh_fwd with dropout on the attention probabilities (csrc/attention_dropout.cu),
    dim_head 32, 64 or 128, any n >= 1.  lse is that of the undropped scores."""
    _req_cuda(qkv)
    inner = heads * dim_head
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous() and qkv.shape == (batch * n, 3 * inner)
    if out is None:
        out = torch.empty((batch * n, inner), dtype=torch.bfloat16, device=qkv.device)
    if lse is None:
        lse = torch.empty((batch, heads, n), dtype=torch.float32, device=qkv.device)
    check(_lib.load().m3l_attention_dropout_fwd(ptr(qkv), batch, n, heads, dim_head, C.c_float(scale),
                                                *_drop_args(dropout), ptr(out), ptr(lse), current_stream()),
          "m3l_attention_dropout_fwd")
    return out, lse


def attention_dropout_bwd(qkv, out, dout, lse, batch, n, heads, dim_head, scale, dropout: Dropout, *, dqkv=None,
                          delta=None):
    """Backward of attention_dropout_fwd (same mask; delta optional as in attention_long_bwd)."""
    _req_cuda(qkv, out, dout, lse, dqkv, delta)
    if dqkv is None:
        dqkv = torch.empty_like(qkv)
    assert dout.is_contiguous() and out.is_contiguous()
    assert delta is None or (delta.dtype == torch.float32 and delta.is_contiguous() and delta.shape == (batch * n, heads))
    check(_lib.load().m3l_attention_dropout_bwd(ptr(qkv), ptr(out), ptr(dout), ptr(lse), ptr(delta), batch, n, heads,
                                                dim_head, C.c_float(scale), *_drop_args(dropout), ptr(dqkv),
                                                current_stream()), "m3l_attention_dropout_bwd")
    return dqkv


def dropout_bwd(dy, dropout: Dropout, *, out=None, colsum=None):
    """out = Z o dy (bf16 [rows, cols], contiguous): the backward of a dropout site of the GEMM epilogues;
    colsum (fp32 [cols]) += column sums of out when given (the bias gradient of the Linear before the dropout)."""
    _req_cuda(dy, out, colsum)
    assert dy.dtype == torch.bfloat16 and dy.is_contiguous() and dy.dim() == 2
    if out is None:
        out = torch.empty_like(dy)
    assert out.shape == dy.shape and out.dtype == torch.bfloat16 and out.is_contiguous()
    assert colsum is None or (colsum.dtype == torch.float32 and colsum.numel() == dy.shape[1])
    check(_lib.load().m3l_dropout_bwd(ptr(dy), dy.shape[0], dy.shape[1], *_drop_args(dropout), ptr(out), ptr(colsum),
                                      current_stream()), "m3l_dropout_bwd")
    return out


# longest sequence the single-CTA kernels of csrc/attention.cu take; above it csrc/attention_long.cu runs
SHORT_ATTENTION_MAX_N = 256
# head widths with kernels: 64 (attention.cu / attention_long.cu), 32 and 128 (attention_dh.cu)
ATTENTION_HEAD_DIMS = (32, 64, 128)


def _mha_kernels(n, dim_head):
    if dim_head != 64:
        return attention_dh_fwd, attention_dh_bwd
    if n <= SHORT_ATTENTION_MAX_N:
        return attention_fwd, attention_bwd
    return attention_long_fwd, attention_long_bwd


def mha_fwd(qkv, batch, n, heads, dim_head, scale, *, out=None, lse=None, dropout: Optional[Dropout] = None):
    """Multi-head attention forward for any sequence length.  64-wide heads: attention_fwd up to
    SHORT_ATTENTION_MAX_N tokens, attention_long_fwd above; 32- and 128-wide heads: attention_dh_fwd for every n;
    with dropout, attention_dropout_fwd for every n and width.
    The one place the model code picks between the kernel families."""
    if dropout is not None:
        return attention_dropout_fwd(qkv, batch, n, heads, dim_head, scale, dropout, out=out, lse=lse)
    f = _mha_kernels(n, dim_head)[0]
    return f(qkv, batch, n, heads, dim_head, scale, out=out, lse=lse)


def mha_bwd(qkv, out, dout, lse, batch, n, heads, dim_head, scale, *, dqkv=None, delta=None,
            dropout: Optional[Dropout] = None):
    """Backward of mha_fwd (same selection by n, dim_head and dropout)."""
    if dropout is not None:
        return attention_dropout_bwd(qkv, out, dout, lse, batch, n, heads, dim_head, scale, dropout, dqkv=dqkv,
                                     delta=delta)
    f = _mha_kernels(n, dim_head)[1]
    return f(qkv, out, dout, lse, batch, n, heads, dim_head, scale, dqkv=dqkv, delta=delta)


# ------------------------------------------------------------------------------------------
# optimizer
# ------------------------------------------------------------------------------------------
def grad_sumsq(grads, state):
    check(_lib.load().m3l_grad_sumsq(ptr(grads), C.c_size_t(grads.numel()), ptr(state), current_stream()),
          "m3l_grad_sumsq")


OPT_STATE_DOUBLES = 8     # step, sumsq, total norm, 1 - beta1^t, sqrt(1 - beta2^t), spare


def optimizer_step_begin(state, betas=(0.9, 0.999), hyper=None):
    assert state.numel() >= 5 and state.dtype == torch.float64
    check(_lib.load().m3l_optimizer_step_begin(ptr(state), C.c_float(betas[0]), C.c_float(betas[1]), ptr(hyper),
                                               current_stream()), "m3l_optimizer_step_begin")


def clip_adamw(params, grads, exp_avg, exp_avg_sq, state, *, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01,
               max_norm=0.5, write_clipped_grad=True, hyper=None):
    """hyper: optional device fp32 [6] = [lr, beta1, beta2, eps, weight_decay, max_norm] read at run time (graph replay)."""
    check(_lib.load().m3l_clip_adamw(ptr(params), ptr(grads), ptr(exp_avg), ptr(exp_avg_sq),
                                     C.c_size_t(params.numel()), ptr(state), C.c_float(lr), C.c_float(betas[0]),
                                     C.c_float(betas[1]), C.c_float(eps), C.c_float(weight_decay),
                                     C.c_float(max_norm), int(write_clipped_grad), ptr(hyper), current_stream()),
          "m3l_clip_adamw")


def ema_update(teacher, student, beta: float):
    """teacher = teacher * beta + (1 - beta) * student, in place, over flat fp32 tensors."""
    _req_cuda(teacher, student)
    assert teacher.dtype == torch.float32 and student.dtype == torch.float32 and teacher.numel() == student.numel()
    assert teacher.is_contiguous() and student.is_contiguous()
    check(_lib.load().m3l_ema_update(ptr(teacher), ptr(student), C.c_size_t(teacher.numel()), C.c_float(beta),
                                     C.c_float(1.0 - beta), current_stream()), "m3l_ema_update")


def cast_bf16(src, dst):
    check(_lib.load().m3l_cast_bf16(ptr(src), ptr(dst), C.c_size_t(src.numel()), current_stream()), "m3l_cast_bf16")


def transpose_cast_bf16(src_base, dst_base, descs_dev, count):
    check(_lib.load().m3l_transpose_cast_bf16(ptr(src_base), ptr(dst_base), ptr(descs_dev), count,
                                              current_stream()), "m3l_transpose_cast_bf16")


def layerscale_fold(w, b, gamma, wf, wf_t=None, bf=None):
    """wf = bf16(gamma[:, None] * w) (gamma None: bf16(w)), wf_t = its transpose, bf = gamma * b, all in place
    (w fp32 [rows, cols]; rounded exactly as torch rounds the same expression)."""
    _req_cuda(w, b, gamma, wf, wf_t, bf)
    rows, cols = w.shape
    assert w.dtype == torch.float32 and w.is_contiguous()
    assert wf.dtype == torch.bfloat16 and wf.is_contiguous() and wf.shape == (rows, cols)
    assert wf_t is None or (wf_t.dtype == torch.bfloat16 and wf_t.is_contiguous() and wf_t.shape == (cols, rows))
    for v in (b, gamma, bf):
        assert v is None or (v.dtype == torch.float32 and v.is_contiguous() and v.numel() == rows)
    check(_lib.load().m3l_layerscale_fold(ptr(w), ptr(b), ptr(gamma), rows, cols, ptr(wf), ptr(wf_t), ptr(bf),
                                          current_stream()), "m3l_layerscale_fold")


def layerscale_unfold(dwf, dbf, w, b, gamma, dw, db, dgamma):
    """Gradients of (w, b, gamma) from those of the folded Linear (w' = gamma o w, b' = gamma o b): dw = gamma o dwf,
    db = gamma o dbf, dgamma = rowsum(w o dwf) + b o dbf (all fp32, written)."""
    _req_cuda(dwf, dbf, w, b, gamma, dw, db, dgamma)
    rows, cols = w.shape
    for m in (dwf, w, dw):
        assert m.dtype == torch.float32 and m.is_contiguous() and m.shape == (rows, cols)
    for v in (dbf, b, gamma, db, dgamma):
        assert v.dtype == torch.float32 and v.is_contiguous() and v.numel() == rows
    check(_lib.load().m3l_layerscale_unfold(ptr(dwf), ptr(dbf), ptr(w), ptr(b), ptr(gamma), rows, cols, ptr(dw),
                                            ptr(db), ptr(dgamma), current_stream()), "m3l_layerscale_unfold")


# ------------------------------------------------------------------------------------------
# launch accounting (bench.py reports how many of our kernels run per step)
# ------------------------------------------------------------------------------------------
_launches = 0
_orig_check = check


def _counting_check(status, what):
    global _launches
    _launches += 1
    _orig_check(status, what)


class LaunchCounter:
    """Counts C-ABI kernel launches issued inside the `with` block (each ops.* call = one launch)."""

    def __enter__(self):
        global check, _launches
        self._start = _launches
        check = _counting_check
        return self

    def __exit__(self, *exc):
        global check
        self.count = _launches - self._start
        check = _orig_check
        return False
