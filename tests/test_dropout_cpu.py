"""CPU: the dropout mask definition (numpy Philox against the Random123 known answers, keep fraction, independence of
keys / sites / planes), the oracle transformer with masks against vit_pytorch's Transformer with its Dropout layers
replaced by the same masks (float64, forward and gradients), the C-ABI of the dropout entry points (exports,
argument errors, fakes), and the compiled dropout attention kernels (tcgen05 / TMA from the uniform datapath, no
spills)."""
import ctypes
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from tests import _dropout_ref as R


@pytest.mark.parametrize("ctr,key,out", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, out):
    got = R.philox4x32_10(np.array(ctr, dtype=np.uint32), key)
    assert tuple(int(v) for v in got) == out


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_keep_fraction(p):
    z = R.mask(0x123456789ABCDEF, 7, 1024, 1024, p)
    thr, scale = R.threshold(p)
    q = 1 - thr / 65536
    n = z.size
    kept = np.count_nonzero(z)
    assert abs(kept / n - q) <= 5 * np.sqrt(q * (1 - q) / n), (kept / n, q)
    assert set(np.unique(z).tolist()) == {0.0, float(scale)}


def test_p_zero_keeps_everything():
    z = R.mask(99, 3, 300, 77, 0.0)
    assert np.all(z == 1.0)


def test_masks_of_different_keys_sites_planes_are_uncorrelated():
    rows, cols, p = 512, 512, 0.5
    base = R.mask(1, 5, rows, cols, p) > 0
    others = [R.mask(2, 5, rows, cols, p), R.mask(1, 6, rows, cols, p), R.mask(1, 5, rows, cols, p, plane=1),
              R.mask(1 << 40, 5, rows, cols, p)]
    for o in others:
        c = np.corrcoef(base.ravel().astype(np.float64), (o > 0).ravel().astype(np.float64))[0, 1]
        assert abs(c) < 5 / np.sqrt(base.size), c
    # the 8 elements served by one Philox call are not correlated either
    u = R.uniforms(1, 5, rows, cols).astype(np.float64)
    for e in range(1, 8):
        c = np.corrcoef(u[:, 0::8].ravel(), u[:, e::8].ravel())[0, 1]
        assert abs(c) < 5 / np.sqrt(u[:, 0::8].size), (e, c)


class _FixedMask(torch.nn.Module):
    def __init__(self, z):
        super().__init__()
        self.z = z

    def forward(self, t):
        return t * self.z


def test_oracle_drop_hook_equals_module_with_fixed_masks():
    """The oracle transformer with a drop hook = vit_pytorch.vit.Transformer (the stub the reference imports) whose
    nn.Dropout layers multiply by the same fixed masks; float64, forward and every gradient."""
    from oracle.stubs.vit_pytorch.vit import Transformer as VitTransformer
    torch.manual_seed(0)
    B, n, dim, depth, heads, dh, mlp = 2, 13, 32, 2, 2, 16, 48
    m = VitTransformer(dim, depth, heads, dh, mlp, dropout=0.3).double()
    hook = R.MaskHook(key=0xDEADBEEF12345, p=0.3)
    x = torch.randn(B, n, dim, dtype=torch.float64)
    # fixed masks in the module, from the same hook
    for l, (attn, ff) in enumerate(m.layers):
        attn.dropout = _FixedMask(hook.z(l, 0, torch.zeros(B, heads, n, n, dtype=torch.float64)))
        attn.to_out[1] = _FixedMask(hook.z(l, 1, torch.zeros(B, n, dim, dtype=torch.float64)))
        ff.net[3] = _FixedMask(hook.z(l, 2, torch.zeros(B, n, mlp, dtype=torch.float64)))
        ff.net[5] = _FixedMask(hook.z(l, 3, torch.zeros(B, n, dim, dtype=torch.float64)))
    m.train()
    sd = {"t." + k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()
          if not k.endswith(".z")}
    x1, x2 = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    y1 = m(x1)
    y2 = R.transformer(x2, sd, "t", depth, heads, dh, drop=hook)
    assert torch.allclose(y1, y2, rtol=0, atol=1e-12)
    w = torch.randn_like(y1)
    (y1 * w).sum().backward()
    (y2 * w).sum().backward()
    assert torch.allclose(x1.grad, x2.grad, rtol=0, atol=1e-12)
    named = dict(m.named_parameters())
    for k, v in sd.items():
        assert torch.allclose(named[k[2:]].grad, v.grad, rtol=0, atol=1e-12), k
    # without a hook the helper is the oracle itself, bit for bit
    from oracle.vtmae_oracle import transformer as oracle_transformer
    with torch.no_grad():
        assert torch.equal(R.transformer(x, sd, "t", depth, heads, dh), oracle_transformer(x, sd, "t", depth, heads, dh))


# ---------------------------------------------------------------------------------------------- C-ABI
@pytest.fixture(scope="module")
def lib():
    from m3l_b200 import build
    path = build.build(verbose=False)
    lib = ctypes.CDLL(str(path))
    lib.m3l_last_error.restype = ctypes.c_char_p
    return lib


_SYMS = ("m3l_attention_dropout_fwd", "m3l_attention_dropout_bwd", "m3l_dropout_bwd")


def test_dropout_symbols_are_declared_and_exported(lib):
    from m3l_b200 import _lib
    header = (Path(__file__).resolve().parents[1] / "include" / "m3l_b200.h").read_text()
    for sym in _SYMS:
        assert sym in _lib.EXPORTED_SYMBOLS
        assert re.search(rf"\bint {sym}\(", header), sym
        assert hasattr(lib, sym)


_D = ctypes.c_void_p(16)          # never dereferenced: the argument checks come first
_FD = ctypes.cast(_D, ctypes.POINTER(ctypes.c_float))
_F = ctypes.c_float


def _fwd(lib, key, p, dh=64):
    return lib.m3l_attention_dropout_fwd(_D, 1, 300, 4, dh, _F(0.125), key, 1, _F(p), _D, _FD, None)


def _bwd(lib, key, p, dh=64):
    return lib.m3l_attention_dropout_bwd(_D, _D, _D, _FD, None, 1, 300, 4, dh, _F(0.125), key, 1, _F(p), _D, None)


def _elt(lib, key, p):
    return lib.m3l_dropout_bwd(_D, 10, 24, key, 1, _F(p), _D, None, None)


@pytest.mark.parametrize("call", [_fwd, _bwd, _elt])
def test_dropout_argument_errors(lib, call):
    assert call(lib, None, 0.1) == 1
    assert b"null dropout key" in lib.m3l_last_error()
    for p in (-0.1, 1.0, 1.5, float("nan"), 1.0 - 2.0 ** -18):
        assert call(lib, _D, p) == 1, p
        assert b"outside [0, 1)" in lib.m3l_last_error()


@pytest.mark.parametrize("dh", [16, 48, 96, 256])
def test_dropout_attention_rejects_other_widths(lib, dh):
    assert _fwd(lib, _D, 0.1, dh) == 3
    assert b"dim_head" in lib.m3l_last_error()
    assert _bwd(lib, _D, 0.1, dh) == 3
    assert b"dim_head" in lib.m3l_last_error()


def test_gemm_rejects_dropout_on_other_epilogues(lib):
    from m3l_b200 import _lib
    def args(**kw):
        a = _lib.GemmArgs()
        a.a = a.b = a.out = 16
        a.lda = a.ldb = a.ldo = 64
        a.m, a.n, a.k = 128, 64, 64
        a.splits, a.alpha = 1, 1.0
        a.drop_key, a.drop_site, a.drop_p = 16, 1, 0.1
        for k, v in kw.items():
            setattr(a, k, v)
        return a
    bad = [dict(), dict(out_mode=1), dict(act=2, aux_in=16, ld_aux=64), dict(act=3), dict(act=1, residual=16, ldr=64),
           dict(residual=16, ldr=64, dot_side=16, ld_dot=64, dot_out=16)]
    for kw in bad:
        assert lib.m3l_gemm_bf16(ctypes.byref(args(**kw)), None) == 1, kw
    assert lib.m3l_gemm_bf16(ctypes.byref(args(residual=16, ldr=64, drop_key=None)), None) == 1
    assert b"null dropout key" in lib.m3l_last_error()
    assert lib.m3l_gemm_bf16(ctypes.byref(args(residual=16, ldr=64, drop_p=1.0)), None) == 1
    assert b"outside [0, 1)" in lib.m3l_last_error()


def test_dropout_fakes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    import m3l_b200.torch_ops as T
    assert {"attention_dropout_fwd", "attention_dropout_bwd", "dropout_bwd"} <= set(T.registered_ops())
    OPS = torch.ops.m3l
    B, n, H, dh = 3, 257, 4, 32
    with FakeTensorMode():
        qkv = torch.empty(B * n, 3 * H * dh, dtype=torch.bfloat16, device="cuda")
        key = torch.empty(1, dtype=torch.int64, device="cuda")
        o, lse = OPS.attention_dropout_fwd(qkv, B, n, H, dh, dh ** -0.5, key, 4, 0.1)
        assert o.shape == (B * n, H * dh) and o.dtype == torch.bfloat16
        assert lse.shape == (B, H, n) and lse.dtype == torch.float32
        d = OPS.attention_dropout_bwd(qkv, o, o, lse, B, n, H, dh, dh ** -0.5, key, 4, 0.1)
        assert d.shape == qkv.shape and d.dtype == torch.bfloat16
        y = torch.empty(70000, 13, dtype=torch.bfloat16, device="cuda")
        z = OPS.dropout_bwd(y, key, 3, 0.5)
        assert z.shape == y.shape and z.dtype == torch.bfloat16


# ---------------------------------------------------------------------------------------------- compiled code
def _sass(obj):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).exists():
        pytest.skip("cuobjdump not available")
    return subprocess.run([cuobjdump, "-sass", str(obj)], capture_output=True, text=True).stdout.splitlines()


def test_dropout_attention_sass_is_tcgen05_from_the_uniform_datapath(lib):
    from m3l_b200 import build
    sass = _sass(build.OBJ / "attention_dropout.o")
    text = "\n".join(sass)
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in text, mnemonic
    issue = [i for i, l in enumerate(sass) if re.search(r"\b(UTCHMMA|UTMALDG|UTMASTG|UTMAREDG)\b", l)]
    bad = [i for i in issue if any("BRA.U.ANY" in l for l in sass[i + 1:i + 4])]
    assert not bad, f"{len(bad)} of {len(issue)} MMA / TMA instructions are issued from a waterfall loop"


def test_dropout_attention_kernels_do_not_spill(lib):
    from m3l_b200 import build
    log = (build.OBJ / "attention_dropout.ptxas.log").read_text()
    kernels = re.findall(r"Function properties for (\S*attn_long_drop_\S*)\n\s*(\d+) bytes stack frame, "
                         r"(\d+) bytes spill stores", log)
    assert len(kernels) == 9, log          # per width: forward, dK / dV backward, dQ backward
    for width in ("Li32E", "Li64E", "Li128E"):
        assert sum(width in name for name, _, _ in kernels) == 3, width
    for name, _, spill in kernels:
        assert spill == "0", name

