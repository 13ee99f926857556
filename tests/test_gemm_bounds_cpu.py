"""CPU: the float64 GEMM / feed-forward-block reference of tests/_gemm_ref.py is right (against torch float64 matmul,
F.gelu and its autograd, F.layer_norm and its autograd), its budgets are finite, non-negative and shaped like their
outputs, an fp32 emulation that rounds where the kernels round stays inside them on every input family, the Python
mirror of the host's kernel selection reproduces the selections the other tests document, and the case table of
tests/test_gemm_bounds_gpu.py reaches every GEMM kernel the built library contains."""
import math
import re
import shutil
import subprocess
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

from tests import _gemm_cases as K
from tests import _gemm_ref as G

DEV = "cpu"


def _side(M, N, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(N, generator=g, dtype=torch.float64).float(),
            torch.randn(M, N, generator=g, dtype=torch.float64).bfloat16(),
            (torch.rand(M, N, generator=g, dtype=torch.float64) * 1.2 - 0.1).bfloat16())


# ------------------------------------------------------------------------------------------ reference vs torch
@pytest.mark.parametrize("M,N,K", [(1, 8, 8), (33, 72, 200), (129, 264, 64)])
def test_reference_matches_torch(M, N, K):
    a, b = G.make_operands("randn", M, N, K, 1, DEV)
    bias, res, aux = _side(M, N, 2)
    A, B = a.double(), b.double()
    z = A @ B.t() + bias.double()
    r = G.gemm_reference(a, b, bias=bias, residual=res)
    torch.testing.assert_close(r.want["out"], z + res.double(), rtol=1e-13, atol=1e-13)
    zz = z.clone().requires_grad_(True)
    F.gelu(zz).backward(torch.ones_like(zz))
    r = G.gemm_reference(a, b, bias=bias, act=1)
    torch.testing.assert_close(r.want["out"], F.gelu(z), rtol=1e-13, atol=1e-13)
    torch.testing.assert_close(r.want["aux"], zz.grad, rtol=1e-12, atol=1e-13)
    r = G.gemm_reference(a, b, act=2, aux_in=aux)
    torch.testing.assert_close(r.want["out"], (A @ B.t()) * aux.double(), rtol=1e-13, atol=1e-13)
    r = G.gemm_reference(a, b, bias=bias, act=3)
    torch.testing.assert_close(r.want["out"], z.clamp(min=0), rtol=1e-13, atol=1e-13)
    init = torch.randn(M, N, dtype=torch.float64).float()
    r = G.gemm_reference(a.t().contiguous(), b.t().contiguous(), mn_major=True, init=init, splits=3)
    torch.testing.assert_close(r.want["out"], init.double() + A @ B.t(), rtol=1e-13, atol=1e-13)
    o = (A @ B.t()).bfloat16()
    dot, _ = G.rowdot_reference(o[:, :64 * (N // 64)], res[:, :64 * (N // 64)]) if N >= 64 else (None, None)
    if dot is not None:
        torch.testing.assert_close(dot, (o.double() * res.double())[:, :64 * (N // 64)].view(M, -1, 64).sum(-1))


def test_ln_bwd_reference_matches_layer_norm_autograd():
    M, Kd = 37, 200
    a, b = G.make_operands("randn", M, 256, Kd, 3, DEV)
    x = torch.randn(M, 256, dtype=torch.float64).bfloat16()
    gamma = (torch.rand(256, dtype=torch.float64) + 0.5).float()
    skip = torch.randn(M, 256, dtype=torch.float64).bfloat16()
    X = x.double()
    mean, var = X.mean(1, keepdim=True), X.var(1, unbiased=False, keepdim=True)
    stats = torch.cat([mean, 1 / torch.sqrt(var + 1e-5)], 1)
    r = G.ln_bwd_reference(a, b, x, stats, gamma, skip)
    xr = X.clone().requires_grad_(True)
    gr = gamma.double().requires_grad_(True)
    br = torch.zeros(256, dtype=torch.float64, requires_grad=True)
    dy = a.double() @ b.double().t()
    F.layer_norm(xr, (256,), gr, br, eps=1e-5).backward(dy)
    torch.testing.assert_close(r.want["dx"], xr.grad + skip.double(), rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(r.want["dgamma"], gr.grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(r.want["dbeta"], br.grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(r.want["dx_colsum"], (xr.grad + skip.double()).sum(0), rtol=1e-10, atol=1e-10)


def test_ln_mlp_reference_matches_torch():
    M, H = 19, 384
    g = torch.Generator().manual_seed(4)
    x = torch.randn(M, 256, generator=g, dtype=torch.float64).bfloat16()
    w1 = (torch.randn(H, 256, generator=g, dtype=torch.float64) / 16).bfloat16()
    w2 = (torch.randn(256, H, generator=g, dtype=torch.float64) / 20).bfloat16()
    gm, bt = torch.rand(256, generator=g, dtype=torch.float64).float() + 0.5, torch.randn(256, generator=g).float() * .1
    b1, b2 = torch.randn(H, generator=g).float() * .1, torch.randn(256, generator=g).float() * .1
    r = G.ln_mlp_reference(x, gm, bt, w1, b1, w2, b2, 1e-5)
    X = x.double()
    y = F.layer_norm(X, (256,), gm.double(), bt.double(), eps=1e-5)
    want = X + F.linear(F.gelu(F.linear(y, w1.double(), b1.double())), w2.double(), b2.double())
    torch.testing.assert_close(r.want["out"], want, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------ budgets
CASES_CPU = [K.Case(33, 136, 200, bias=True, res="res"), K.Case(31, 72, 56, act=1, bias=True),
             K.Case(129, 264, 8, act=2), K.Case(65, 120, 264, f32=True, bias=True),
             K.Case(40, 72, 129, mn=True, splits=3), K.Case(33, 256, 768, ln="skip")]


@pytest.mark.parametrize("family", G.FAMILIES)
@pytest.mark.parametrize("c", CASES_CPU, ids=lambda c: c.id)
def test_budgets_are_finite_and_non_negative(family, c):
    for name, want, budget in _refs(c, family):
        assert torch.isfinite(budget).all() and (budget >= 0).all(), name
        assert budget.shape == want.shape, name


def _refs(c, family, emulated=None):
    a, b = G.make_operands(family, c.M, c.N, c.K, 5, DEV, mn_major=c.mn)
    bias, res, aux = _side(c.M, c.N, 6)
    if c.ln:
        x = torch.randn(c.M, 256, dtype=torch.float64)
        X = x.bfloat16()
        stats = torch.cat([x.mean(1, keepdim=True), 1 / torch.sqrt(x.var(1, unbiased=False, keepdim=True) + 1e-5)],
                          1).float()
        gm = (torch.rand(256, dtype=torch.float64) + 0.5).float()
        r = G.ln_bwd_reference(a, b, X, stats, gm, res)
        got = _emulate_ln_bwd(a, b, X, stats, gm, res) if emulated else None
        return [(k, r.want[k], r.budget[k]) + ((got[k],) if got else ()) for k in ("dx", "dgamma", "dbeta", "dx_colsum")]
    init = torch.randn(c.M, c.N, dtype=torch.float64).float() if c.mn else None
    kw = dict(mn_major=c.mn, bias=bias if c.bias else None, residual=res if c.res else None, act=c.act,
              aux_in=aux if c.act == 2 else None, init=init, splits=c.splits)
    r = G.gemm_reference(a, b, **kw)
    got = _emulate_gemm(a, b, out_f32=c.f32, **kw) if emulated else None
    return [(k, r.want[k], r.budget[k]) + ((got[k],) if got else ()) for k in r.want]


# ------------------------------------------------------------------------------------------ fp32 emulation
def _acc16(A, B):
    """fp32 accumulation in 16-term steps (each step's exact sum rounded once onto the running fp32 value)."""
    Kd = A.shape[1]
    acc = torch.zeros(A.shape[0], B.shape[0], dtype=torch.float32)
    for k0 in range(0, Kd, 16):
        acc = (acc.double() + A[:, k0:k0 + 16] @ B[:, k0:k0 + 16].t()).float()
    return acc


def _perturb(x, rel, seed):
    g = torch.Generator().manual_seed(seed)
    s = torch.randint(0, 2, x.shape, generator=g).float() * 2 - 1
    return (x.double() * (1 + s.double() * rel)).float()


def _gelu_pair32(x):
    """gelu_pair in fp32, with the reciprocal and the exponential off by their documented approximation errors."""
    ax = x.abs()
    den = ax * torch.tensor(0.3275911 * 0.70710678118654752, dtype=torch.float32) + 1
    t = _perturb(1.0 / den, 2.0 ** -23, 1)
    ea = x * x * torch.tensor(-0.5 * 1.4426950408889634, dtype=torch.float32)
    e = _perturb(torch.exp2(ea), 2.0 ** -22, 2)
    q = torch.full_like(x, -0.5 * 1.061405429)
    for c in (0.5 * 1.453152027, -0.5 * 1.421413741, 0.5 * 0.284496736, -0.5 * 0.254829592):
        q = q * t + c
    nu = q * t * e
    sg = torch.where(x < 0, -1.0, 1.0).float()
    cdf = sg * nu + (sg * 0.5 + 0.5)
    return x * cdf, x * e * torch.tensor(0.39894228040143268, dtype=torch.float32) + cdf


def _emulate_gemm(a, b, *, mn_major, bias, residual, act, aux_in, init, splits, out_f32):
    A, B = G.operands64(a, b, mn_major)
    acc = _acc16(A, B)
    if init is not None:
        return {"out": init + acc}
    v = acc + bias if bias is not None else acc
    if act == 3:
        v = v.clamp(min=0)
    if act == 1:
        h, g = _gelu_pair32(v)
        return {"out": h.bfloat16(), "aux": g.bfloat16()}
    if act == 2:
        v = v * aux_in.float()
    if residual is not None:
        v = v + residual.float()
    return {"out": v if out_f32 else v.bfloat16()}


def _emulate_ln_bwd(a, b, x, stats, gamma, skip):
    dy = _acc16(a.double(), b.double())
    mean, rstd = stats[:, 0:1], stats[:, 1:2]
    xh = (x.float() - mean) * rstd
    g = dy * gamma
    c1 = g.sum(1, keepdim=True) * (1 / 256)
    c2 = (g * xh).sum(1, keepdim=True) * (1 / 256)
    dx = rstd * (g - c1 - xh * c2) + skip.float()
    return {"dx": dx.bfloat16(), "dgamma": (dy * xh).sum(0), "dbeta": dy.sum(0), "dx_colsum": dx.sum(0)}


@pytest.mark.parametrize("family", G.FAMILIES)
@pytest.mark.parametrize("c", CASES_CPU, ids=lambda c: c.id)
def test_fp32_emulation_stays_inside_the_budget(family, c):
    for name, want, budget, got in _refs(c, family, emulated=True):
        g2, w2, b2 = (got, want, budget) if got.dim() == 2 else (got[None], want[None], budget[None])
        r, msg = G.ratio(name, g2, w2, b2)
        assert r <= 1.0, msg


@pytest.mark.parametrize("family", ["randn", "smallvar", "offset"])
def test_ln_mlp_fp32_emulation_stays_inside_the_budget(family):
    M, H = 40, 256
    g = torch.Generator().manual_seed(9)
    x = torch.randn(M, 256, generator=g, dtype=torch.float64)
    x = {"smallvar": 0.03 * x, "offset": 4 + 0.05 * x}.get(family, x).bfloat16()
    w1 = (torch.randn(H, 256, generator=g, dtype=torch.float64) / 16).bfloat16()
    w2 = (torch.randn(256, H, generator=g, dtype=torch.float64) / 16).bfloat16()
    gm, bt = (torch.rand(256, generator=g, dtype=torch.float64) + 0.5).float(), torch.randn(256, generator=g) * .1
    b1, b2 = torch.randn(H, generator=g) * .1, torch.randn(256, generator=g) * .1
    X = x.float()
    mean = X.sum(1, keepdim=True) * (1 / 256)
    var = torch.clamp((X * X).sum(1, keepdim=True) * (1 / 256) - mean * mean, min=0)
    rstd = _perturb(torch.rsqrt(var + 1e-5), 2.0 ** -22, 3)
    xn = ((X * rstd + (-mean * rstd)) * gm + bt).bfloat16()
    pre = _acc16(xn.double(), w1.double()) + b1
    na = torch.clamp(-pre.abs(), min=G.RB_CLAMP)
    eh = _perturb(torch.exp2(G._rb_poly(na.double()).float()), 2.0 ** -22, 4)
    h = (pre.clamp(min=0) + na * eh).bfloat16()
    y = (_acc16(h.double(), w2.double()) + b2)
    for two, out in ((False, (X + y).bfloat16()), (True, (X.double() + y.bfloat16().double()).float().bfloat16())):
        r = G.ln_mlp_reference(x, gm, bt, w1, b1, w2, b2, 1e-5, two_roundings=two)
        rr, msg = G.ratio("out", out, r.want["out"], r.budget["out"])
        assert rr <= 1.0, msg
    r = G.ln_mlp_reference(x, gm, bt, w1, b1, w2, b2, 1e-5, saved=(torch.cat([mean, rstd], 1), xn, h, None))
    for name, got in (("mean", mean), ("rstd", rstd), ("xn", xn), ("h", h)):
        rr, msg = G.ratio(name, got, r.want[name], r.budget[name])
        assert rr <= 1.0, msg


# ------------------------------------------------------------------------------------------ selection and coverage
@pytest.mark.parametrize("shape,kw,want", [
    ((49152, 768, 256), {}, (256, False, False, 0, True)),
    ((31232, 192, 256), dict(out_mode=1), (128, False, False, 3, True)),
    ((49152, 1024, 256), dict(act=1), ("gelu16",)),
    ((49152, 1024, 256), dict(act=1, colsum=True), (256, False, False, 1, True)),
    ((49152, 256, 1024), dict(ln=True), (256, False, False, 5, False)),
    ((2560, 256, 256), dict(residual=True), (128, False, False, 0, False)),
    ((256, 768, 49152), dict(mn_major=True, splits=8, bn=256), (256, True, True, 4, False)),
])
def test_mirror_reproduces_documented_selections(shape, kw, want):
    assert G.select_kernel(*shape, 148, **kw) == want


def test_mirror_clamps_splits():
    assert G.clamp_splits(200, 64) == 4 and G.clamp_splits(1000, 64) == 16 and G.clamp_splits(320, 4) == 3


def _library_kernels():
    from m3l_b200 import build as B
    lib = B.LIB if B.LIB.exists() else B.build(verbose=False)
    tool = shutil.which("cuobjdump") or str(Path(B.NVCC).parent / "cuobjdump")
    elf = subprocess.run([tool, "-elf", str(lib)], capture_output=True, text=True, check=True).stdout
    names = sorted({m for m in re.findall(r"\.text\.(_Z\S+)", elf)})
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return {G.parse_kernel_name(n) for n in dem.splitlines()} - {None}


def test_case_table_covers_every_gemm_kernel_in_the_library():
    built = _library_kernels()
    gemm = {k for k in built if k[0] not in ("gelu16", "ln_mlp")}
    assert len(gemm) == 28 and ("gelu16",) in built and {("ln_mlp", False), ("ln_mlp", True)} <= built, \
        sorted(map(G.variant_label, built))
    reached = {c.kernel(K.B200_SMS) for c in K.CASES}
    reached |= {("ln_mlp", save) for _, _, _, save, _ in K.LN_MLP}
    missing = sorted(map(G.variant_label, built - reached))
    assert not missing, f"kernels without a case in tests/_gemm_cases.py: {missing}"
    print(f"{len(gemm)} gemm_bf16_kernel + gemm_gelu16 + 2 ln_mlp instantiations, all reached by "
          f"{len(K.CASES)} cases")


def test_model_shapes_are_derived():
    cs = K.model_cases()
    assert any(c.N == 1536 and c.act == 2 and c.colsum for c in cs)          # DINOv2 GELU' with the bias gradient
    assert any(c.K == 592 for c in cs) and any(c.M == 49152 and c.N == 768 for c in cs)
    assert all(math.gcd(c.M if c.mn else c.K, 8) == 8 for c in cs)          # row pitches the tensor maps accept
