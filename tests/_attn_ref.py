"""Float64 reference of multi-head attention, forward and backward, in the kernels' layouts, with an elementwise error
budget for every output derived from where the kernels round.

Layouts (those of m3l_attention_fwd / _bwd and their long / dh variants):
    qkv  [B*n, 3*H*dh] bf16, columns [q | k | v], head h at columns h*dh .. (h+1)*dh of each third
    dout, out [B*n, H*dh];  lse [B, H, n];  dqkv like qkv;  delta [B*n, H] = rowsum(dout * out) per head

Rounding points of the kernels (csrc/attention.cu, csrc/attention_long.cuh):
    S = Q K^T               fp32 accumulation of exact bf16 x bf16 products on the tensor core
    p = exp(S*scale - m)    approximate exp2 (fast math) of an fp32 argument; m = row max (forward, n <= 256), a
                            lagging running max (forward, long kernels) or the saved LSE (backward)
    P V, P^T dO             P rounded to bf16, fp32 accumulation;  O = (P V) / rowsum(p) in fp32, stored as bf16
    lse = m + log(sum p)    approximate logarithm, fp32
    dP = dO V^T             fp32;  delta = rowsum(dO * out) from the bf16 out (or rowsum(p * dP), n <= 16)
    dS = p (dP - delta) scale, rounded to bf16;  dQ = dS K, dK = dS^T Q, dV = P^T dO in fp32, stored as bf16

The budget of a bf16 output Y is E, the error its fp32 value may carry into the final rounding: an element passes when
some value within E of Y rounds to it, and its ratio is the smallest such error over E (0 for the correctly rounded
value, above 1 for anything no admissible fp32 result rounds to).  lse is fp32 and its budget bounds |error| directly.
Inside the kernels, a bf16 operand x (P, dS) computed with error e is off by at most rb(x, e), the largest distance from
x to what a value in [x - e, x + e] rounds to (round to nearest is monotone: the two ends give it).  E is built from
these bounds (u = 2^-8 is bf16's unit roundoff, 2^-24 fp32's):
    es   = (dh/16 + 3) 2^-23 * scale * max_j sum_d |q_d k_jd|      absolute error of a scaled score: the dh/16 tensor
           core steps round (or truncate, hence 2^-23 per step) once each, plus three roundings of the fp32 operands
    ef   = 2 es + 2^-21 max_j |S_j| + 2^-22 T                        relative error of a forward exponential: the score
           and the row max each off by es, the fp32 argument (scale, log2 e, max subtracted) rounded at most 8 times
           relative to the largest scaled score, and 2^-22 for the approximate exp2 (and, in the long kernels, for
           each of the T = ceil(n / 128) key tiles' approximate rescale factors)
    eb   = es + |lse_kernel - lse| + 2^-21 (max_j |S_j| + |lse|) + 2^-22        the same for the backward's exponentials,
           which subtract the forward's LSE
    kacc(m) = (ceil(m/16) + 1 + T) 2^-23                          relative error of an m-term fp32 tensor-core
           contraction (one rounding per 16-term step, the rescales of the long kernels' accumulator)
    1e-5 for the approximate logarithm: __logf is lg2.approx times ln 2, documented to within 2^-21.4 absolute on
           [0.5, 2] and a few ulp elsewhere, about 1.5e-6 for the sums here (log(sum) <= log(n) < 6); rounded up.
The forward's P in the long kernels is scaled by a running max the reference does not follow, so there its rounding
is bounded by the plain u |p|.  Every first-order bound above is multiplied by the safety factor C = 2 before it is
propagated.  Nothing here is fitted to observed errors: an element outside its budget is a defect.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import torch

C = 2.0                       # safety factor on every first-order error bound
U = 2.0 ** -8                 # bf16 unit roundoff
LOG_ALLOWANCE = 1e-5          # approximate logarithm (see the module docstring)
FLUSH = 2.0 ** -125           # fast-math exponentials flush results below the normal range to zero


def is_long(n, dh):
    """True when mha_fwd/bwd run csrc/attention_long.cuh (online softmax over 128-key tiles) for (n, dh)."""
    return not (dh == 64 and n <= 256)


def rb(y, e):
    """Largest |bf16(x) - y| over fp32 x in [y - e, y + e] (round to nearest even through fp32, as the kernels do)."""
    lo = (y - e).float().bfloat16().double()
    hi = (y + e).float().bfloat16().double()
    return torch.maximum((lo - y).abs(), (hi - y).abs())


def _rounded(x, e):
    """Error bound of bf16(x') for a value x' within e of x, including a flush to zero of tiny values."""
    return torch.maximum(rb(x, e), torch.where(x.abs() < FLUSH, x.abs() + e, torch.zeros_like(x)))


def split_qkv(qkv, B, n, H, dh):
    """[B*n, 3*H*dh] -> q, k, v [B, H, n, dh] (float64)."""
    q, k, v = qkv.double().view(B, n, 3, H, dh).permute(2, 0, 3, 1, 4)
    return q, k, v


def heads_view(x, B, n, H, dh):
    """[B*n, H*dh] -> [B, H, n, dh]."""
    return x.view(B, n, H, dh).transpose(1, 2)


@dataclass
class Reference:
    out: torch.Tensor          # [B, H, n, dh] float64 (also dq, dk, dv)
    lse: torch.Tensor          # [B, H, n]
    delta: torch.Tensor        # [B, H, n] rowsum(dout * out)
    dq: torch.Tensor
    dk: torch.Tensor
    dv: torch.Tensor
    budget: dict = field(default_factory=dict)   # same keys, same shapes: elementwise |error| bounds


def forward_reference(qkv, B, n, H, dh, scale):
    """Exact forward in float64: dict of q, k, v, S (scaled scores), m (row max), pt = exp(S - m), l = rowsum(pt),
    P, out, lse, and the forward error budgets of out and lse."""
    q, k, v = split_qkv(qkv, B, n, H, dh)
    S = (q @ k.transpose(-1, -2)) * scale
    m = S.amax(-1, keepdim=True)
    pt = torch.exp(S - m)
    l = pt.sum(-1, keepdim=True)
    P = pt / l
    out = P @ v
    lse = (m + torch.log(l)).squeeze(-1)
    long = is_long(n, dh)
    T = math.ceil(n / 128) if long else 1
    es = (dh / 16 + 3) * 2.0 ** -23 * scale * (q.abs() @ k.abs().transpose(-1, -2)).amax(-1, keepdim=True)
    smax = S.abs().amax(-1, keepdim=True)
    ef = C * (2 * es + 2.0 ** -21 * smax + 2.0 ** -22 * T)
    kacc = lambda m_: (math.ceil(m_ / 16) + 1 + T) * 2.0 ** -23
    if long:
        Rf = (U * (1 + ef) + ef) * pt
    else:
        Rf = _rounded(pt, ef * pt)
    PV = P @ v.abs()
    b_out = (Rf @ v.abs()) / l + C * kacc(n) * PV + (ef + C * (n * 2.0 ** -24 + 2.0 ** -23)) * out.abs()
    b_lse = C * (es + ef + n * 2.0 ** -24 + LOG_ALLOWANCE + 2.0 ** -23 * (smax + lse.abs().unsqueeze(-1))).squeeze(-1)
    return dict(q=q, k=k, v=v, S=S, m=m, pt=pt, l=l, P=P, out=out, lse=lse, es=es, smax=smax, T=T, kacc=kacc,
                b_out=b_out, b_lse=b_lse)


def reference(qkv, dout, B, n, H, dh, scale, *, out=None, lse=None):
    """Float64 forward and backward of softmax(q k^T * scale) v for every (sample, head), with error budgets.

    out, lse: the kernel's forward outputs that its backward is given.  The backward's budgets then use their actual
    errors (lse) and the actual rounding of the delta computed from the bf16 out; without them they use the forward
    budgets instead."""
    f = forward_reference(qkv, B, n, H, dh, scale)
    q, k, v, S, P, O = f["q"], f["k"], f["v"], f["S"], f["P"], f["out"]
    es, smax, kacc = f["es"], f["smax"], f["kacc"]
    do = heads_view(dout.double(), B, n, H, dh)
    dP = do @ v.transpose(-1, -2)
    delta = (do * O).sum(-1)
    dS = P * (dP - delta.unsqueeze(-1)) * scale
    dv = P.transpose(-1, -2) @ do
    dq = dS @ k
    dk = dS.transpose(-1, -2) @ q

    dL = (lse.double() - f["lse"]).abs() if lse is not None else f["b_lse"]
    eb = C * (es + dL.unsqueeze(-1) + 2.0 ** -21 * (smax + f["lse"].abs().unsqueeze(-1)) + 2.0 ** -22)
    Rb = _rounded(P, eb * P)
    edP = C * (dh / 16 + 1) * 2.0 ** -23 * (do.abs() @ v.abs().transpose(-1, -2))
    # delta: from the bf16 out (tcgen05 and long kernels, and callers that pass it) or as rowsum(p * dP) (n <= 16)
    o_used = heads_view(out.double(), B, n, H, dh) if out is not None else O
    d_from_out = (do * o_used).sum(-1)
    D_out = (d_from_out - delta).abs() if out is not None else (do.abs() * ((1 + U) * f["b_out"] + U * O.abs())).sum(-1)
    D_out = D_out + C * dh * 2.0 ** -24 * (do * o_used).abs().sum(-1)
    PdP = (P * dP.abs()).sum(-1)
    D_p = (eb.squeeze(-1) + C * n * 2.0 ** -24) * PdP + (P * edP).sum(-1) * (1 + eb.squeeze(-1))
    Dd = (D_out + D_p).unsqueeze(-1)
    E_ds = scale * (eb * P * (dP - delta.unsqueeze(-1)).abs() + P * (1 + eb) * (edP + Dd)) + C * 2.0 ** -22 * dS.abs()
    Rds = _rounded(dS, E_ds)
    kq = kacc(n)
    E_dv = Rb.transpose(-1, -2) @ do.abs() + C * kq * ((P + Rb).transpose(-1, -2) @ do.abs())
    A = dS.abs() + Rds
    E_dq = Rds @ k.abs() + C * kq * (A @ k.abs())
    E_dk = Rds.transpose(-1, -2) @ q.abs() + C * kq * (A.transpose(-1, -2) @ q.abs())
    budget = dict(out=f["b_out"], lse=f["b_lse"], dv=E_dv, dq=E_dq, dk=E_dk)
    return Reference(out=O, lse=f["lse"], delta=delta, dq=dq, dk=dk, dv=dv, budget=budget)


def cell_distance(got, want):
    """Distance from want (float64) to the interval of reals that round to nearest to the bf16 value got: the
    smallest error before the rounding that explains got (exact to within fp32's half ulp at the interval's ends)."""
    g = got.double()
    mant, ex = torch.frexp(g)                                   # |g| = |mant| 2^ex, |mant| in [0.5, 1)
    above = torch.ldexp(torch.ones_like(g), ex - 8)             # bf16 spacing above |g|; below it halves at 2^k
    below = torch.where(mant.abs() == 0.5, above / 2, above)
    tiny = 2.0 ** -133                                          # bf16's subnormal spacing (and that of zero)
    above, below = above.clamp(min=tiny), below.clamp(min=tiny)
    lo = torch.where(g >= 0, g - below / 2, g - above / 2)
    hi = torch.where(g >= 0, g + above / 2, g + below / 2)
    return torch.maximum(torch.maximum(lo - want, want - hi), torch.zeros_like(g))


def worst_ratio(name, got, want, budget):
    """Largest error / budget over every element, with where it occurs.  got, want, budget: [B, H, n(, dh)].  A bf16
    got is measured by cell_distance (the error its fp32 value must have had), an fp32 one by |got - want|.
    Returns (ratio, message); a non-finite element, or an error where the budget is zero, gives ratio inf."""
    err = cell_distance(got, want) if got.dtype == torch.bfloat16 else (got.double() - want).abs()
    got = got.double()
    ratio = torch.where(budget > 0, err / torch.where(budget > 0, budget, torch.ones_like(budget)),
                        torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    ratio = torch.where(torch.isfinite(got), ratio, torch.full_like(ratio, math.inf))
    idx = int(ratio.flatten().argmax())
    where = list(torch.unravel_index(torch.tensor(idx), ratio.shape))
    labels = ("b", "h", "row", "col")
    loc = ", ".join(f"{l}={int(i)}" for l, i in zip(labels, where))
    r = float(ratio.flatten()[idx])
    msg = (f"{name}: worst |err| / budget = {r:.3g} at ({loc}): got {float(got.flatten()[idx]):.6g}, "
           f"want {float(want.flatten()[idx]):.6g}, budget {float(budget.flatten()[idx]):.3g}")
    return r, msg


# ------------------------------------------------------------------------------------------ input families
FAMILIES = ("randn", "x4", "x8", "negative", "constant", "dominant0", "dominant_last")


def make_inputs(family, B, n, H, dh, scale, seed=0, device="cuda"):
    """qkv [B*n, 3*H*dh] and dout [B*n, H*dh] (bf16) of one input family:
        randn          q, k, v, dout ~ N(0, 1)
        x4, x8         the same times 4 / 8: large scores, a nearly one-hot softmax
        negative       q = a u + noise, k = -a u + noise along a shared direction u, with scale * a^2 = 40: every real
                       scaled score is about -40, so a padded key (score exactly 0) that leaks in dominates its row
        constant       every key of a (sample, head) equal: constant scores, uniform P
        dominant0      key 0 (dominant_last: key n - 1) is a u with scale * a^2 = 24 and every query leans along u:
                       P is one-hot on it.  dout is +-v of that key plus a little noise, so dP of the dominant key
                       equals delta and dS ~ 0 there: an error in P or in delta is not hidden under dS's own rounding
    """
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(B, n, 3, H, dh, generator=g, dtype=torch.float64)
    dout = torch.randn(B, n, H, dh, generator=g, dtype=torch.float64)
    u = torch.nn.functional.normalize(torch.randn(H, dh, generator=g, dtype=torch.float64), dim=-1)
    if family == "x4":
        x = x * 4
    elif family == "x8":
        x = x * 8
    elif family == "negative":
        a = math.sqrt(40 / scale)
        x[:, :, 0] += a * u
        x[:, :, 1] += -a * u
    elif family == "constant":
        x[:, :, 1] = x[:, :1, 1]
    elif family in ("dominant0", "dominant_last"):
        j = 0 if family == "dominant0" else n - 1
        a = math.sqrt(24 / scale)
        x[:, :, 0] = 0.5 * x[:, :, 0] + a * u
        x[:, j, 1] = a * u
        sign = torch.randint(0, 2, (B, n, H, 1), generator=g).double() * 2 - 1
        dout = sign * x[:, j:j + 1, 2].bfloat16().double() + 0.1 * dout
    elif family != "randn":
        raise ValueError(family)
    qkv = x.reshape(B * n, 3 * H * dh).to(device).bfloat16().contiguous()
    return qkv, dout.reshape(B * n, H * dh).to(device).bfloat16().contiguous()
