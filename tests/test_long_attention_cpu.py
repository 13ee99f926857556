"""CPU: the long-sequence attention entry points (csrc/attention_long.cu) are exported and reject bad arguments with a
message, their torch.library fakes give the right shapes, and the compiled kernels are tcgen05 / TMA code that issues
from the uniform datapath and does not spill."""
import ctypes
import re
import shutil
import subprocess
from pathlib import Path

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from m3l_b200 import build
    path = build.build(verbose=False)
    lib = ctypes.CDLL(str(path))
    lib.m3l_last_error.restype = ctypes.c_char_p
    return lib


def test_long_attention_symbols_are_exported(lib):
    from m3l_b200 import _lib
    for sym in ("m3l_attention_long_fwd", "m3l_attention_long_bwd"):
        assert sym in _lib.EXPORTED_SYMBOLS
        assert hasattr(lib, sym)


def test_long_attention_rejects_bad_arguments(lib):
    f = ctypes.c_float(0.125)
    assert lib.m3l_attention_long_fwd(None, 1, 300, 4, 64, f, None, None, None) == 1
    assert b"null" in lib.m3l_last_error()
    assert lib.m3l_attention_long_bwd(None, None, None, None, None, 1, 300, 4, 64, f, None, None) == 1
    assert b"null" in lib.m3l_last_error()
    dummy = ctypes.c_void_p(16)        # never dereferenced: the argument checks come first
    fdummy = ctypes.cast(dummy, ctypes.POINTER(ctypes.c_float))
    assert lib.m3l_attention_long_fwd(dummy, 1, 300, 4, 32, f, dummy, fdummy, None) == 3
    assert b"dim_head" in lib.m3l_last_error()
    assert lib.m3l_attention_long_bwd(dummy, dummy, dummy, fdummy, None, 1, 300, 4, 128, f, dummy, None) == 3
    assert b"dim_head" in lib.m3l_last_error()
    assert lib.m3l_attention_long_fwd(dummy, 1, 0, 4, 64, f, dummy, fdummy, None) == 1
    assert b"n/heads/batch" in lib.m3l_last_error()


def test_long_attention_fakes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    import m3l_b200.torch_ops as T
    assert {"attention_long_fwd", "attention_long_bwd"} <= set(T.registered_ops())
    OPS = torch.ops.m3l
    B, n, H = 3, 1374, 6
    with FakeTensorMode():
        qkv = torch.empty(B * n, 3 * H * 64, dtype=torch.bfloat16, device="cuda")
        o, lse = OPS.attention_long_fwd(qkv, B, n, H, 64, 0.125)
        assert o.shape == (B * n, H * 64) and o.dtype == torch.bfloat16
        assert lse.shape == (B, H, n) and lse.dtype == torch.float32
        d = OPS.attention_long_bwd(qkv, o, o, lse, B, n, H, 64, 0.125)
        assert d.shape == qkv.shape and d.dtype == torch.bfloat16


def _sass(obj):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).exists():
        pytest.skip("cuobjdump not available")
    return subprocess.run([cuobjdump, "-sass", str(obj)], capture_output=True, text=True).stdout.splitlines()


def test_long_attention_sass_is_tcgen05_from_the_uniform_datapath(lib):
    from m3l_b200 import build
    sass = _sass(build.OBJ / "attention_long.o")
    text = "\n".join(sass)
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in text, mnemonic
    issue = [i for i, l in enumerate(sass) if re.search(r"\b(UTCHMMA|UTMALDG|UTMASTG|UTMAREDG)\b", l)]
    bad = [i for i in issue if any("BRA.U.ANY" in l for l in sass[i + 1:i + 4])]
    assert not bad, f"{len(bad)} of {len(issue)} MMA / TMA instructions are issued from a waterfall loop"


def test_long_attention_kernels_do_not_spill(lib):
    from m3l_b200 import build
    log = (build.OBJ / "attention_long.ptxas.log").read_text()
    kernels = re.findall(r"Function properties for (\S*attn_long_\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores",
                         log)
    assert len(kernels) == 3, log         # forward, dK / dV backward, dQ backward
    for name, _, spill in kernels:
        assert spill == "0", name
