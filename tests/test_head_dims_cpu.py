"""CPU: the 32- / 128-wide-head attention entry points (csrc/attention_dh.cu) are exported and reject bad arguments
with a message, their torch.library fakes give the right shapes, the compiled kernels are tcgen05 / TMA code that
issues from the uniform datapath and does not spill, the 64-wide kernels of attention_long.o are instruction for
instruction what they were before the kernels became a template on the head width, and the transformer modules
accept exactly the head widths that have kernels."""
import ctypes
import re
import shutil
import subprocess
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def lib():
    from m3l_b200 import build
    path = build.build(verbose=False)
    lib = ctypes.CDLL(str(path))
    lib.m3l_last_error.restype = ctypes.c_char_p
    return lib


def test_head_dim_symbols_are_exported(lib):
    from m3l_b200 import _lib
    for sym in ("m3l_attention_dh_fwd", "m3l_attention_dh_bwd"):
        assert sym in _lib.EXPORTED_SYMBOLS
        assert hasattr(lib, sym)


def test_head_dim_attention_rejects_bad_arguments(lib):
    f = ctypes.c_float(0.125)
    assert lib.m3l_attention_dh_fwd(None, 1, 300, 4, 32, f, None, None, None) == 1
    assert b"null" in lib.m3l_last_error()
    assert lib.m3l_attention_dh_bwd(None, None, None, None, None, 1, 300, 4, 128, f, None, None) == 1
    assert b"null" in lib.m3l_last_error()
    dummy = ctypes.c_void_p(16)        # never dereferenced: the argument checks come first
    fdummy = ctypes.cast(dummy, ctypes.POINTER(ctypes.c_float))
    for n, heads, batch in ((0, 4, 1), (300, 0, 1), (300, 4, -1)):
        assert lib.m3l_attention_dh_fwd(dummy, batch, n, heads, 32, f, dummy, fdummy, None) == 1
        assert b"n/heads/batch" in lib.m3l_last_error()
        assert lib.m3l_attention_dh_bwd(dummy, dummy, dummy, fdummy, None, batch, n, heads, 128, f, dummy, None) == 1
        assert b"n/heads/batch" in lib.m3l_last_error()


@pytest.mark.parametrize("dh", [16, 48, 64, 96, 256])
def test_head_dim_attention_rejects_other_widths(lib, dh):
    f = ctypes.c_float(0.125)
    dummy = ctypes.c_void_p(16)
    fdummy = ctypes.cast(dummy, ctypes.POINTER(ctypes.c_float))
    assert lib.m3l_attention_dh_fwd(dummy, 1, 300, 4, dh, f, dummy, fdummy, None) == 3
    assert b"dim_head" in lib.m3l_last_error()
    assert lib.m3l_attention_dh_bwd(dummy, dummy, dummy, fdummy, None, 1, 300, 4, dh, f, dummy, None) == 3
    assert b"dim_head" in lib.m3l_last_error()


@pytest.mark.parametrize("dh", [32, 128])
def test_head_dim_attention_fakes(dh):
    from torch._subclasses.fake_tensor import FakeTensorMode
    import m3l_b200.torch_ops as T
    assert {"attention_dh_fwd", "attention_dh_bwd"} <= set(T.registered_ops())
    OPS = torch.ops.m3l
    B, n, H = 3, 1374, 6
    with FakeTensorMode():
        qkv = torch.empty(B * n, 3 * H * dh, dtype=torch.bfloat16, device="cuda")
        o, lse = OPS.attention_dh_fwd(qkv, B, n, H, dh, dh ** -0.5)
        assert o.shape == (B * n, H * dh) and o.dtype == torch.bfloat16
        assert lse.shape == (B, H, n) and lse.dtype == torch.float32
        d = OPS.attention_dh_bwd(qkv, o, o, lse, B, n, H, dh, dh ** -0.5)
        assert d.shape == qkv.shape and d.dtype == torch.bfloat16


def _sass(obj):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).exists():
        pytest.skip("cuobjdump not available")
    return subprocess.run([cuobjdump, "-sass", str(obj)], capture_output=True, text=True).stdout.splitlines()


def test_head_dim_sass_is_tcgen05_from_the_uniform_datapath(lib):
    from m3l_b200 import build
    sass = _sass(build.OBJ / "attention_dh.o")
    text = "\n".join(sass)
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in text, mnemonic
    issue = [i for i, l in enumerate(sass) if re.search(r"\b(UTCHMMA|UTMALDG|UTMASTG|UTMAREDG)\b", l)]
    bad = [i for i in issue if any("BRA.U.ANY" in l for l in sass[i + 1:i + 4])]
    assert not bad, f"{len(bad)} of {len(issue)} MMA / TMA instructions are issued from a waterfall loop"


def test_head_dim_kernels_do_not_spill(lib):
    from m3l_b200 import build
    log = (build.OBJ / "attention_dh.ptxas.log").read_text()
    kernels = re.findall(r"Function properties for (\S*attn_long_\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores",
                         log)
    assert len(kernels) == 6, log         # per width: forward, dK / dV backward, dQ backward
    for width in ("Li32E", "Li128E"):
        assert sum(width in name for name, _, _ in kernels) == 3, width
    for name, _, spill in kernels:
        assert spill == "0", name


# normalised SASS (tools/sass_normalise.py) of attention_long.o as built from attention_long.cu before the kernels
# became a template on the head width, and the nvcc that built it
_DH64_SASS_SHA256 = "5bf292ebb5648a7f9760dca40032d06820a823fc9156cd0da69fc2ff0de5bbc3"
_DH64_SASS_NVCC = "12.9"


def test_dh64_kernels_are_unchanged_by_the_template(lib):
    from m3l_b200 import build
    ver = subprocess.run([build.NVCC, "--version"], capture_output=True, text=True).stdout
    if f"release {_DH64_SASS_NVCC}," not in ver:
        pytest.skip(f"reference digest was taken with nvcc {_DH64_SASS_NVCC}")
    if not (shutil.which("cuobjdump") or Path("/usr/local/cuda/bin/cuobjdump").exists()):
        pytest.skip("cuobjdump not available")
    sys.path.insert(0, str(ROOT / "tools"))
    try:
        import sass_normalise
    finally:
        sys.path.pop(0)
    kernels = sass_normalise.normalised_sass(build.OBJ / "attention_long.o")
    assert sorted(kernels) == ["attn_long_bwd_kernel<0>", "attn_long_bwd_kernel<1>", "attn_long_fwd_kernel"]
    assert sass_normalise.digest(build.OBJ / "attention_long.o") == _DH64_SASS_SHA256


@pytest.mark.parametrize("dh", [32, 64, 128])
def test_transformer_accepts_supported_head_widths(dh):
    from m3l_b200.vtmae import Transformer
    t = Transformer(256, 1, 256 // dh, dh, 512)
    assert t.dim_head == dh and t.layers[0][0].to_qkv.weight.shape == (3 * 256, 256)


@pytest.mark.parametrize("dh", [16, 48, 96])
def test_transformer_rejects_other_head_widths(dh):
    from m3l_b200._lib import M3LError
    from m3l_b200.vtmae import Transformer
    with pytest.raises(M3LError, match=r"\(32, 64, 128\)"):
        Transformer(256, 1, 4, dh, 512)
