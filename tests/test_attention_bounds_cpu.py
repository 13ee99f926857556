"""CPU: the float64 attention reference of tests/_attn_ref.py is right (against torch's scaled_dot_product_attention and
autograd), its error budgets are finite and non-negative, and an fp32 emulation that rounds where the kernels round
stays inside them, on every input family."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests import _attn_ref as R

DEV = "cpu"


@pytest.mark.parametrize("B,n,H,dh", [(2, 1, 2, 64), (2, 17, 3, 64), (1, 130, 2, 64), (2, 40, 2, 32), (1, 33, 1, 128)])
def test_reference_matches_sdpa_and_autograd(B, n, H, dh):
    scale = dh ** -0.5
    qkv, dout = R.make_inputs("randn", B, n, H, dh, scale, seed=1, device=DEV)
    ref = R.reference(qkv, dout, B, n, H, dh, scale)
    q, k, v = (t.clone().requires_grad_(True) for t in R.split_qkv(qkv, B, n, H, dh))
    o = F.scaled_dot_product_attention(q, k, v, scale=scale)
    do = R.heads_view(dout.double(), B, n, H, dh)
    o.backward(do)
    torch.testing.assert_close(ref.out, o.detach(), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(ref.dq, q.grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(ref.dk, k.grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(ref.dv, v.grad, rtol=1e-10, atol=1e-12)
    lse = torch.logsumexp((q @ k.transpose(-1, -2)).detach() * scale, -1)
    torch.testing.assert_close(ref.lse, lse, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(ref.delta, (do * o.detach()).sum(-1), rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("family", R.FAMILIES)
def test_budgets_are_finite_and_non_negative(family):
    B, n, H, dh = 2, 37, 2, 64
    qkv, dout = R.make_inputs(family, B, n, H, dh, dh ** -0.5, seed=2, device=DEV)
    ref = R.reference(qkv, dout, B, n, H, dh, dh ** -0.5)
    for name, b in ref.budget.items():
        assert torch.isfinite(b).all() and (b >= 0).all(), name
        assert b.shape == getattr(ref, name).shape, name


def _emulate(qkv, dout, B, n, H, dh, scale):
    """The kernels' arithmetic in fp32 with their bf16 rounding points (csrc/attention.cu): returns out, lse, dq, dk,
    dv in the reference's [B, H, n(, dh)] layout, the delta of the backward taken from the bf16 out."""
    q, k, v = qkv.float().view(B, n, 3, H, dh).permute(2, 0, 3, 1, 4)
    do = dout.float().view(B, n, H, dh).transpose(1, 2)
    log2e = 1.4426950408889634
    sl2 = torch.tensor(scale * log2e, dtype=torch.float32)
    s = q @ k.transpose(-1, -2)
    mx = s.amax(-1, keepdim=True)
    p = torch.exp2(s * sl2 - mx * sl2)
    l = p.sum(-1, keepdim=True)
    out = ((p.bfloat16().float() @ v) * (1.0 / l)).bfloat16()
    lse = (mx * scale + torch.log(l)).squeeze(-1)
    pb = torch.exp2(s * sl2 - (lse * log2e).unsqueeze(-1))
    dp = do @ v.transpose(-1, -2)
    delta = (do * out.float()).sum(-1, keepdim=True)
    ds = (pb * (dp - delta) * scale).bfloat16().float()
    dv = (pb.bfloat16().float().transpose(-1, -2) @ do).bfloat16()
    dq = (ds @ k).bfloat16()
    dk = (ds.transpose(-1, -2) @ q).bfloat16()
    return out, lse, dq, dk, dv


CASES = [(f, 64 ** -0.5) for f in R.FAMILIES] + [("randn", 1.0), ("randn", 0.01)]


@pytest.mark.parametrize("family,scale", CASES)
@pytest.mark.parametrize("n,dh", [(1, 64), (10, 64), (17, 64), (129, 64), (256, 64), (70, 32), (70, 128)])
def test_fp32_emulation_stays_inside_the_budget(family, scale, n, dh):
    B, H = 2, 2
    if dh != 64:
        scale = scale * math.sqrt(64 / dh)
    qkv, dout = R.make_inputs(family, B, n, H, dh, scale, seed=3, device=DEV)
    out, lse, dq, dk, dv = _emulate(qkv, dout, B, n, H, dh, scale)
    out_flat = out.transpose(1, 2).reshape(B * n, H * dh)
    ref = R.reference(qkv, dout, B, n, H, dh, scale, out=out_flat, lse=lse)
    for name, got in (("out", out), ("lse", lse), ("dq", dq), ("dk", dk), ("dv", dv)):
        r, msg = R.worst_ratio(name, got, getattr(ref, name), ref.budget[name])
        assert r <= 1.0, msg


def test_worst_ratio_reports_the_location():
    want = torch.zeros(2, 3, 4, 5, dtype=torch.float64)
    got = want.clone()
    got[1, 2, 3, 4] = 0.5
    r, msg = R.worst_ratio("lse", got, want, torch.full_like(want, 0.1))
    assert r == pytest.approx(5.0) and "b=1, h=2, row=3, col=4" in msg
    got[0, 0, 0, 0] = math.nan
    assert R.worst_ratio("lse", got, want, torch.full_like(want, 0.1))[0] == math.inf
    # bf16: the error that must have preceded the rounding.  0.5 is reached from anything above 0.5 - 2^-10.
    r, _ = R.worst_ratio("dq", got[1:].bfloat16(), want[1:], torch.full_like(want[1:], 0.1))
    assert r == pytest.approx((0.5 - 2.0 ** -10) / 0.1)
    want = torch.full((1, 1, 1, 2), 1.0 + 2.0 ** -10, dtype=torch.float64)
    assert R.worst_ratio("out", want.bfloat16(), want, torch.zeros_like(want))[0] == 0.0    # correctly rounded
    up = (want + 2.0 ** -7).bfloat16()                        # 1 + 2^-7, reached from 1 + 2^-8 up: 0.75 * 2^-8 away
    assert R.worst_ratio("out", up, want, torch.full_like(want, 2.0 ** -8))[0] == pytest.approx(0.75)
    assert R.worst_ratio("out", up, want, torch.full_like(want, 2.0 ** -9))[0] == pytest.approx(1.5)


def test_cell_distance_never_exceeds_the_error_before_rounding():
    g = torch.Generator().manual_seed(5)
    y = torch.randn(100000, generator=g, dtype=torch.float64) * 10.0 ** torch.randint(-6, 6, (100000,), generator=g)
    e = y.abs() * 2.0 ** -torch.randint(4, 20, (100000,), generator=g).double()
    x = y + (torch.rand(100000, generator=g, dtype=torch.float64) * 2 - 1) * e
    d = R.cell_distance(x.float().bfloat16(), y)
    # x is rounded through fp32 on its way to bf16, which may move it by fp32's half ulp
    assert (d <= e + 2.0 ** -24 * x.abs()).all()
    assert (R.cell_distance(y.float().bfloat16(), y) <= 2.0 ** -24 * y.abs()).all()
