"""ctypes binding of the in-tree C-ABI library (include/m3l_b200.h).

There is no CPU fallback: if the shared object is missing, or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

# M3L_B200_LIB: development override (A/B runs of kernel variants built next to the shipped library)
_LIB_PATH = Path(os.environ.get("M3L_B200_LIB") or (Path(__file__).resolve().parent / "lib" / "libm3l_b200.so"))
_lib = None


class M3LError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("b", C.c_void_p),
        ("lda", C.c_int32), ("ldb", C.c_int32),
        ("a_mn_major", C.c_int32), ("b_mn_major", C.c_int32),
        ("m", C.c_int32), ("n", C.c_int32), ("k", C.c_int32),
        ("splits", C.c_int32), ("bn", C.c_int32),
        ("out", C.c_void_p), ("ldo", C.c_int32), ("out_mode", C.c_int32),
        ("bias", C.c_void_p), ("residual", C.c_void_p), ("ldr", C.c_int32),
        ("act", C.c_int32), ("aux_out", C.c_void_p), ("aux_in", C.c_void_p),
        ("ld_aux", C.c_int32), ("alpha", C.c_float), ("colsum_out", C.c_void_p),
        ("out2", C.c_void_p), ("dot_side", C.c_void_p), ("ld_dot", C.c_int32), ("dot_out", C.c_void_p),
        ("ln_x", C.c_void_p), ("ln_stats", C.c_void_p), ("ln_gamma", C.c_void_p), ("ln_skip", C.c_void_p),
        ("ln_dgamma", C.c_void_p), ("ln_dbeta", C.c_void_p), ("ln_dxcol", C.c_void_p),
        ("drop_key", C.c_void_p), ("drop_site", C.c_int32), ("drop_p", C.c_float),
    ]


class LnMlpArgs(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("rows", C.c_int32), ("dim", C.c_int32), ("hidden", C.c_int32),
        ("gamma", C.c_void_p), ("beta", C.c_void_p), ("eps", C.c_float),
        ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p),
        ("out", C.c_void_p), ("out_has_x", C.c_int32), ("stats", C.c_void_p), ("xn_out", C.c_void_p),
        ("h_out", C.c_void_p), ("gp_out", C.c_void_p),
    ]


def lib_path() -> Path:
    return _LIB_PATH


def load() -> C.CDLL:
    """Loads libm3l_b200.so (building it first if M3L_B200_AUTOBUILD=1 and it is absent)."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        if os.environ.get("M3L_B200_AUTOBUILD", "0") == "1":
            from . import build as _build

            _build.build(verbose=False)
        else:
            raise M3LError(
                f"{_LIB_PATH} not found: the CUDA extension is not built. Run "
                "`python -m m3l_b200.build` (or __graft_entry__.build()); there is no CPU fallback."
            )
    lib = C.CDLL(str(_LIB_PATH))
    lib.m3l_last_error.restype = C.c_char_p
    lib.m3l_last_error.argtypes = []
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().m3l_last_error().decode("utf-8", "replace")
        raise M3LError(f"{what} failed with status {status}: {msg}")


def ptr(t) -> C.c_void_p:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    return C.c_void_p(t.data_ptr())


def current_stream() -> C.c_void_p:
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class MaskSegments(C.Structure):
    _fields_ = [("count", C.c_int32), ("offset", C.c_int32 * 8), ("length", C.c_int32 * 8),
                ("n_masked", C.c_int32 * 8)]


class PatchSource(C.Structure):
    _fields_ = [("src", C.c_void_p * 4), ("channels", C.c_int32), ("height", C.c_int32),
                ("width", C.c_int32), ("patch_h", C.c_int32), ("patch_w", C.c_int32),
                ("token_base", C.c_int32),
                # layout 1: raw-observation addressing (vt_load fused into the patch loads; include/m3l_b200.h)
                ("layout", C.c_int32), ("dtype", C.c_int32), ("stride_b", C.c_int64), ("chan_group", C.c_int32),
                ("stride_f", C.c_int32), ("stride_ch", C.c_int32), ("stride_y", C.c_int32), ("stride_x", C.c_int32),
                ("norm_lo", C.c_float), ("norm_span", C.c_float)]


class MatrixDesc(C.Structure):
    _fields_ = [("src_offset", C.c_int64), ("dst_offset", C.c_int64), ("rows", C.c_int32),
                ("cols", C.c_int32)]


# every symbol include/m3l_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = (
    "m3l_last_error", "m3l_gemm_bf16", "m3l_ln_mlp_fwd", "m3l_mask_indices", "m3l_patch_layernorm", "m3l_layernorm_fwd",
    "m3l_layernorm_bwd", "m3l_decoder_assemble_fwd", "m3l_decoder_assemble_bwd", "m3l_rowclass_sum",
    "m3l_mse_loss", "m3l_colsum", "m3l_ln_param_grad", "m3l_attention_fwd", "m3l_attention_bwd",
    "m3l_attention_long_fwd", "m3l_attention_long_bwd",
    "m3l_attention_dh_fwd", "m3l_attention_dh_bwd", "m3l_attention_dropout_fwd", "m3l_attention_dropout_bwd",
    "m3l_dropout_bwd", "m3l_grad_sumsq", "m3l_optimizer_step_begin", "m3l_clip_adamw", "m3l_cast_bf16",
    "m3l_transpose_cast_bf16", "m3l_layerscale_fold", "m3l_layerscale_unfold", "m3l_token_mean_fwd", "m3l_token_mean_bwd",
    "m3l_im2col", "m3l_col2im_relu", "m3l_token_finish", "m3l_token_finish_bwd", "m3l_vt_load", "m3l_patchify", "m3l_row_scatter_add", "m3l_ema_update",
)
