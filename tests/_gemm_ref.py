"""Float64 reference of the tcgen05 GEMM epilogues (csrc/gemm.cu, csrc/gemm_gelu.cu) and of the fused feed-forward
block (csrc/rowblock.cu, ln_mlp_fwd), with an elementwise error budget for every output derived from where the
kernels round; the host's kernel selection mirrored in Python; the input families.

Layouts are those of ops.gemm: a [M, K], b [N, K] (K-major) or a [K, M], b [K, N] (mn_major, wgrad), out [M, N].

Budgets use the conventions of tests/_attn_ref.py: a bf16 output passes when some value within its budget E rounds to
it (worst_ratio / cell_distance), an fp32 output when |got - want| <= E; every first-order bound carries the safety
factor C = 2; u = 2^-24 is fp32's unit roundoff.  Rounding points, from the kernels:
    acc          fp32 tensor-core accumulation of exact bf16 x bf16 products: kacc(K) S, S = sum_k |a_k b_k|
                 (_attn_ref.kacc_model with no rescales)
    split-K      EPI_F32_RED: `splits` fp32 reduce-adds onto the caller's out, any order: (splits + 1) u (|init| + S)
    bias         one fp32 add: u |acc + bias|
    ReLU         exact and 1-Lipschitz: the budget passes through, the reference is max(pre, 0)
    dropout      kept elements one fp32 multiply by the scale (scale E + u |y|); dropped ones must be exactly 0
    residual     the bf16 side tile added in fp32: u |y|;  GELU' backward: acc * aux_in, one multiply: |aux| E + u |y|
    GELU, GELU'  gelu_pair (common.cuh): Phi from Abramowitz & Stegun 7.1.26 (|erf error| <= 1.5e-7, so 7.5e-8 on Phi),
                 t = rcp.approx(1 + p|x|/sqrt 2) (1 ulp, plus the fma: 1.5 * 2^-23 relative), e = ex2.approx(-x^2 log2e
                 / 2) (2^-22 relative, plus 3 roundings of the argument: 1.5 u x^2 relative), the polynomial in Horner
                 form (5 u sum_i |c_i t^i| absolute, and its sensitivity |sum_i i c_i t^i| / |sum_i c_i t^i| to t), then
                 the products with t, e, the sign fma and x (one u each).  The pre-activation's own error E_x passes
                 through |GELU'| <= 1.13 and |GELU''| <= 0.8.  Exponentials that flush to zero add 2^-120 (1 + |x|).
    row-dot      dot_out: fp32 fma chain over the kernel's bf16 out times dot_side, 64 terms: 64 u sum |o s|
    column sums  colsum_out: fp32 atomics of the kernel's bf16 out over rows < M onto the initial value, any order:
                 (M + 1) u (|init| + sum |out|)
    LN backward  EPI_LN_BWD with the caller's (mean, rstd): xhat = (x - mean) rstd (2 u), g = dy gamma (u), c1 = mean
                 of g over 256 columns (summation depth 36: pairs, 32 sequential groups, the two halves), c2 = mean of
                 g xhat (fma chain, depth 130), dx = fma(rstd, (g - c1) - xhat c2, skip) (4 u), one bf16 rounding;
                 dgamma = sum dy xhat, dbeta = sum dy, dx_colsum = sum of the fp32 dx: atomics over M rows, any order
    ln_mlp       LayerNorm statistics in fp32 (sum and sum of squares: depth 10; mean (u), var = fma(-mean, mean,
                 sq / 256) (u, plus 2 |mean| E_mean), rstd = rsqrt.approx(var + eps) (2^-22 relative, u on the add)),
                 xn = fma(fma(x, rstd, -mean rstd), gamma, beta) (3 u) to bf16; pre = xn W1^T + b1; h = GELU(pre) by the
                 exp2-polynomial gelu2 of rowblock.cu, whose own error (fit and clamp) is evaluated in float64 at each
                 element (plus 10 u of Horner rounding, 2^-22 for ex2.approx, 3 u on the result) to bf16, kept in TMEM and
                 saved as is; out = x + (h W2^T + b2): one bf16 rounding when x is re-read, two when the block output
                 is rounded to bf16 and then reduce-added in bf16 onto out (out=x, out_has_x): there the budget is
                 rb of the block output plus the float64 rounding of the reference's own sum (2^-52 (|x| + |y|)),
                 because the first rounding can use all of rb and the second land exactly on a tie.
Where the kernel saves an intermediate (stats, xn, h, gp) the next stage's reference starts from the kernel's value;
otherwise the intermediate's budget plus its bf16 rounding (rb) is propagated.  Nothing here is fitted to observed
errors: an element outside its budget is a defect.

The "exact" input family uses small integers for every operand, so every product, fp32 partial sum and output of the
epilogues without a transcendental, a dropout scale or a LayerNorm is exact (or rounds once, deterministically, to
bf16): those outputs must match bit for bit, whatever the budgets say.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import torch

from tests._attn_ref import C, FLUSH, cell_distance, kacc_model, rb, worst_ratio  # noqa: F401

U32 = 2.0 ** -24
BM, BK = 128, 64
EPI_BF16, EPI_GELU_FWD, EPI_GELU_BWD, EPI_F32, EPI_F32_RED, EPI_LN_BWD, EPI_GELU_DROP, EPI_BF16_DROP = range(8)


def kacc(K):
    return kacc_model(K, 0)


def ratio(name, got, want, budget):
    return worst_ratio(name, got, want, budget, labels=("row", "col"))


# ------------------------------------------------------------------------------------------ GELU models
AS_P = 0.3275911
AS_COEF = (0.254829592, -0.284496736, 1.421413741, -1.453152027, 1.061405429)     # c_1 .. c_5 of A&S 7.1.26


def phi(x):
    return 0.5 * (1 + torch.special.erf(x / math.sqrt(2)))


def pdf(x):
    return torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)


def gelu(x):
    return x * phi(x)


def gelu_grad(x):
    return phi(x) + x * pdf(x)


def gelu_pair_error(x):
    """Elementwise bounds of the fp32 evaluation errors of gelu_pair (common.cuh) at the exact pre-activation x:
    (E_gelu, E_gelu_grad), first order, before the factor C."""
    ax = x.abs()
    t = 1.0 / (1.0 + AS_P / math.sqrt(2) * ax)
    poly = sum(c * t ** (i + 1) for i, c in enumerate(AS_COEF))                  # = erfc-like polynomial times t
    dpoly = sum((i + 1) * c * t ** (i + 1) for i, c in enumerate(AS_COEF))
    apoly = sum(abs(c) * t ** (i + 1) for i, c in enumerate(AS_COEF))
    e = torch.exp(-0.5 * x * x)
    u = 0.5 * poly * e                                                            # Phi(-|x|) of the A&S formula
    rel_u = (dpoly.abs() / poly.abs()) * 1.5 * 2.0 ** -23 + 5 * U32 * apoly / poly.abs() + 2.0 ** -22 \
        + 1.5 * U32 * x * x + 3 * U32
    cdf = phi(x)
    e_phi = 7.5e-8 + u * rel_u + U32 * cdf + 2.0 ** -120
    e_h = ax * e_phi + U32 * gelu(x).abs() + 2.0 ** -120 * (1 + ax)
    xpdf = (x * pdf(x)).abs()
    e_g = e_phi + xpdf * (2.0 ** -22 + 1.5 * U32 * x * x + 3 * U32) + U32 * gelu_grad(x).abs() + 2.0 ** -120
    return e_h, e_g


# exp2-polynomial GELU of rowblock.cu (gelu2): erfc(z) / 2 = exp2(P(na)), na = max(-|x|, -6.08)
RB_E = (1.1511168561, -4.5908273735e-01, 5.2926736750e-02, 7.7240424434e-03, 6.4775743001e-04, 1.7755137836e-05)
RB_CLAMP = -6.08


def _rb_poly(na):
    t = torch.full_like(na, RB_E[5])
    for c in reversed(RB_E[:5]):
        t = t * na + c
    return t * na - 1.0


def gelu2_error(x):
    """(E_gelu, E_gelu_grad) of rowblock.cu's gelu2 at x, first order, before the factor C: the formula's own error
    (the polynomial fit and the clamp of na), evaluated in float64 at x, plus its fp32 evaluation."""
    ax = x.abs()
    na = torch.clamp(-ax, min=RB_CLAMP)
    eh = torch.exp2(_rb_poly(na))
    pdf_na = torch.exp(-0.5 * na * na) / math.sqrt(2 * math.pi)
    h_f = x.clamp(min=0) + na * eh
    q = eh + na * pdf_na
    g_f = 0.5 + torch.sign(x) * (0.5 - q)
    horner = 10 * U32 * sum(abs(c) * na.abs() ** (i + 1) for i, c in enumerate(RB_E))   # absolute error of P
    e_eh = eh * (2.0 ** -22 + math.log(2) * (horner + U32)) + 2.0 ** -120
    e_h = (h_f - gelu(x)).abs() + ax * e_eh + 3 * U32 * (gelu(x).abs() + ax) + 2.0 ** -120 * (1 + ax)
    e_g = (g_f - gelu_grad(x)).abs() + e_eh + (na * pdf_na).abs() * (2.0 ** -22 + 1.5 * U32 * na * na + 3 * U32) \
        + 4 * U32 + 2.0 ** -120
    return e_h, e_g


GELU_LIP, GELU_GRAD_LIP = 1.13, 0.8


# ------------------------------------------------------------------------------------------ GEMM reference
@dataclass
class Ref:
    want: dict = field(default_factory=dict)     # name -> float64 tensor
    budget: dict = field(default_factory=dict)   # name -> float64 tensor (same shape)
    exact: set = field(default_factory=set)      # names whose result is exactly representable (exact family)


def operands64(a, b, mn_major):
    """A [M, K], B [N, K] in float64."""
    a, b = a.double(), b.double()
    return (a.t(), b.t()) if mn_major else (a, b)


def gemm_reference(a, b, *, mn_major=False, bias=None, residual=None, act=0, aux_in=None, out_f32=False, init=None,
                   splits=1, keep=None, exact=False):
    """Reference of ops.gemm's main outputs: 'out' (and 'aux' = GELU' for act 1).  keep: the float32 dropout mask of
    tests/_dropout_ref.py (0 or the scale) for the dropout epilogues.  init: the caller's fp32 out (accumulate)."""
    A, B = operands64(a, b, mn_major)
    acc = A @ B.t()
    S = A.abs() @ B.abs().t()
    E = C * kacc(A.shape[1]) * S
    r = Ref()
    if init is not None:                                     # EPI_F32_RED
        want = init.double() + acc
        r.want["out"] = want
        r.budget["out"] = E + C * (splits + 1) * U32 * (init.double().abs() + S)
        if exact and float(S.max() + init.double().abs().max()) < 2 ** 24:
            r.exact.add("out")
        return r
    pre = acc
    if bias is not None:
        pre = acc + bias.double()
        E = E + C * U32 * pre.abs()
    if act == 3:
        pre = pre.clamp(min=0)
    lossless = exact and float(S.max()) < 2 ** 24
    if act == 1:
        eh, eg = gelu_pair_error(pre)
        h, g = gelu(pre), gelu_grad(pre)
        Eh, Eg = GELU_LIP * E + C * eh, GELU_GRAD_LIP * E + C * eg
        if keep is not None:
            z = keep.double()
            h, g = h * z, g * z
            Eh, Eg = Eh * z + C * U32 * h.abs(), Eg * z + C * U32 * g.abs()
        r.want.update(out=h, aux=g)
        r.budget.update(out=Eh, aux=Eg)
        return r
    y = pre
    if act == 2:
        s = aux_in.double()
        y = acc * s
        E = E * s.abs() + C * U32 * y.abs()
    if keep is not None:
        z = keep.double()
        y = y * z
        E = E * z + C * U32 * y.abs()
        lossless = False
    if residual is not None:
        y = y + residual.double()
        E = E + C * U32 * y.abs()
    r.want["out"] = y
    r.budget["out"] = E
    if lossless and not (act == 2 and float((acc * aux_in.double()).abs().max()) >= 2 ** 24):
        r.exact.add("out")
    return r


def rowdot_reference(out, side):
    """dot_out [M, N / 64] from the kernel's bf16 out and the bf16 dot_side."""
    M, N = out.shape
    p = (out.double() * side.double()).view(M, N // 64, 64)
    return p.sum(-1), C * 64 * U32 * p.abs().sum(-1)


def colsum_reference(out, init):
    """colsum_out [N] = init + column sums of the kernel's bf16 out."""
    o = out.double()
    want = init.double() + o.sum(0)
    return want, C * (o.shape[0] + 1) * U32 * (init.double().abs() + o.abs().sum(0))


def ln_bwd_reference(a, b, x, stats, gamma, skip=None, inits=None):
    """EPI_LN_BWD: dx (bf16) and the fp32 column sums dgamma, dbeta, dx_colsum (onto inits, a dict of the initial
    values), with the caller's stats [M, 2] = (mean, rstd) used as given."""
    A, B = operands64(a, b, False)
    dy = A @ B.t()
    E_dy = C * kacc(A.shape[1]) * (A.abs() @ B.abs().t())
    mean, rstd = stats[:, 0:1].double(), stats[:, 1:2].double()
    gm = gamma.double()
    xh = (x.double() - mean) * rstd
    E_xh = C * 2 * U32 * xh.abs()
    g = dy * gm
    E_g = gm.abs() * E_dy + C * U32 * g.abs()
    n = x.shape[1]
    c1 = g.mean(1, keepdim=True)
    c2 = (g * xh).mean(1, keepdim=True)
    E_c1 = (E_g.sum(1, keepdim=True) + C * 36 * U32 * g.abs().sum(1, keepdim=True)) / n
    E_c2 = ((E_g * xh.abs() + g.abs() * E_xh).sum(1, keepdim=True) + C * 130 * U32 * (g * xh).abs().sum(1, keepdim=True)) / n
    inner = g - c1 - xh * c2
    E_in = E_g + E_c1 + xh.abs() * E_c2 + c2.abs() * E_xh + C * U32 * ((g - c1).abs() + (xh * c2).abs() + inner.abs())
    dx = rstd * inner + (skip.double() if skip is not None else 0)
    E_dx = rstd * E_in + C * U32 * dx.abs()
    M = x.shape[0]
    r = Ref()
    r.want["dx"], r.budget["dx"] = dx, E_dx
    inits = inits or {}
    for name, t, Et in (("dgamma", dy * xh, E_dy * xh.abs() + dy.abs() * E_xh + C * U32 * (dy * xh).abs()),
                        ("dbeta", dy, E_dy), ("dx_colsum", dx, E_dx)):
        i0 = inits.get(name)
        i0 = i0.double() if i0 is not None else torch.zeros(n, dtype=torch.float64, device=x.device)
        r.want[name] = i0 + t.sum(0)
        r.budget[name] = Et.sum(0) + C * (M + 1) * U32 * (i0.abs() + t.abs().sum(0))
    return r


def ln_mlp_reference(x, gamma, beta, w1, b1, w2, b2, eps, *, saved=None, two_roundings=False):
    """ln_mlp_fwd.  saved = (stats, xn, h, gp) of the kernel (save=True): each stage starts from the kernel's value and
    stats / xn / h / gp are checked too.  two_roundings: the block output is rounded to bf16 and reduce-added in bf16
    onto x (out=x or out_has_x)."""
    X = x.double()
    D = X.shape[1]
    gm, bt = gamma.double(), beta.double()
    mean = X.mean(1, keepdim=True)
    var = X.var(1, unbiased=False, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    E_sum = C * 10 * U32 * X.abs().sum(1, keepdim=True)
    E_mean = E_sum / D + C * U32 * mean.abs()
    E_sq = C * 10 * U32 * (X * X).sum(1, keepdim=True)
    E_var = E_sq / D + 2 * mean.abs() * E_mean + E_mean ** 2 + C * U32 * ((X * X).mean(1, keepdim=True) + var)
    ve = var + eps
    E_ve = E_var + C * U32 * ve
    E_rstd = 0.5 * rstd * E_ve / ve + C * 2.0 ** -22 * rstd
    r = Ref()
    if saved is not None:
        st, xn_k, h_k, gp_k = saved
        r.want["mean"], r.budget["mean"] = mean, E_mean
        r.want["rstd"], r.budget["rstd"] = rstd, E_rstd
        mean, rstd = st[:, 0:1].double(), st[:, 1:2].double()      # the next stage from the kernel's stats
        E_mean = E_rstd = 0.0
    xc = (X - mean) * rstd
    xn = xc * gm + bt
    E_xn = C * U32 * (gm.abs() * (xc.abs() + (mean * rstd).abs()) + xn.abs()) \
        + gm.abs() * ((X - mean).abs() * E_rstd + rstd * E_mean)
    W1, W2 = w1.double(), w2.double()
    if saved is not None:
        r.want["xn"], r.budget["xn"] = xn, E_xn
        XN, R_xn = xn_k.double(), 0.0
    else:
        XN, R_xn = xn, rb(xn, E_xn)
    pre = XN @ W1.t() + b1.double()
    K1 = W1.shape[1]
    E_pre = (R_xn @ W1.abs().t() if saved is None else 0.0) \
        + C * kacc(K1) * ((XN.abs() + R_xn) @ W1.abs().t()) + C * U32 * pre.abs()
    eh, eg = gelu2_error(pre)
    h = gelu(pre)
    E_h = GELU_LIP * E_pre + C * eh
    if saved is not None:
        r.want["h"], r.budget["h"] = h, E_h
        r.want["gp"], r.budget["gp"] = gelu_grad(pre), GELU_GRAD_LIP * E_pre + C * eg
        H, R_h = h_k.double(), 0.0
    else:
        H, R_h = h, rb(h, E_h)
    K2 = W2.shape[1]
    y = H @ W2.t() + b2.double()
    E_y = (R_h @ W2.abs().t() if saved is None else 0.0) + C * kacc(K2) * ((H.abs() + R_h) @ W2.abs().t()) \
        + C * U32 * y.abs()
    if two_roundings:
        # the intermediate rounding can use all of rb and the bf16 sum then land on a tie: the reference's own float64
        # sum X + y (one rounding, 2^-53) is the only slack there
        r.want["out"], r.budget["out"] = X + y, rb(y, E_y) + 2.0 ** -52 * (X.abs() + y.abs())
    else:
        out = X + y
        r.want["out"], r.budget["out"] = out, E_y + C * U32 * out.abs()
    return r


# ------------------------------------------------------------------------------------------ kernel selection
def pick_bn(M, N, sms):
    """gemm_pick_bn (gemm.cu)."""
    tiles_m = (M + BM - 1) // BM
    if N % 256 == 0 and tiles_m * (N // 256) >= sms:
        return 256
    if N >= 128 and tiles_m * ((N + 127) // 128) >= sms // 2:
        return 128
    if N % 128 == 0 and N >= 512:
        return 128
    return 128 if N >= 128 and N % 128 == 0 else 64


def clamp_splits(K, splits):
    kb = (K + BK - 1) // BK
    s = min(max(splits, 1), kb)
    while s > 1 and ((kb + s - 1) // s) * (s - 1) >= kb:
        s -= 1
    return s


def select_kernel(M, N, K, sms, *, bn=0, mn_major=False, splits=1, out_mode=0, act=0, residual=False, dot=False,
                  drop=False, ln=False, colsum=False):
    """The kernel gemm_make_plan / gemm_run launch: ('gelu16',) or (BN, A_MN, B_MN, EPI, WS)."""
    splits = clamp_splits(K, splits)
    kb = (K + BK - 1) // BK
    if ln:
        bn = 256
    if bn == 0:
        bn = pick_bn(M, N, sms)
    tiles_n = (N + bn - 1) // bn
    tiles = ((M + BM - 1) // BM) * tiles_n * splits
    grid = min(tiles, sms)
    ws = (not mn_major and not drop and kb <= 4 and splits == 1 and bn >= 128 and not residual and not dot and act != 2
          and not ln and tiles >= 2 * sms and tiles_n <= grid)
    if ws and bn == 256 and act == 1 and out_mode == 0 and N % 256 == 0 and not colsum:
        return ("gelu16",)
    if mn_major:
        return (bn, True, True, EPI_F32_RED, False)
    if drop:
        return (bn, False, False, EPI_GELU_DROP if act == 1 else EPI_BF16_DROP, False)
    if ws:
        epi = EPI_F32 if out_mode == 1 else EPI_GELU_FWD if act == 1 else EPI_BF16
        return (bn, False, False, epi, True)
    if bn == 256 and ln:
        return (bn, False, False, EPI_LN_BWD, False)
    epi = EPI_F32 if out_mode == 1 else EPI_GELU_FWD if act == 1 else EPI_GELU_BWD if act == 2 else EPI_BF16
    return (bn, False, False, epi, False)


def parse_kernel_name(name):
    """Demangled kernel name -> the key of select_kernel, ('ln_mlp', save) or None for other kernels."""
    import re
    if "gemm_gelu16_kernel" in name:
        return ("gelu16",)
    t = r"(true|false|1|0|\(bool\)1|\(bool\)0)"
    yes = lambda v: v in ("true", "1", "(bool)1")
    m = re.search(r"ln_mlp_fwd_kernel(?:<" + t + r">|ILb([01])E)", name)
    if m:
        return ("ln_mlp", yes(m.group(1) or m.group(2)))
    m = re.search(r"gemm_bf16_kernel<(\d+), " + t + ", " + t + r", (\d+), " + t + ">", name)
    if m:
        return (int(m.group(1)), yes(m.group(2)), yes(m.group(3)), int(m.group(4)), yes(m.group(5)))
    m = re.search(r"gemm_bf16_kernelILi(\d+)ELb([01])ELb([01])ELi(\d+)ELb([01])E", name)      # mangled
    if m:
        return (int(m.group(1)), yes(m.group(2)), yes(m.group(3)), int(m.group(4)), yes(m.group(5)))
    return None


def variant_label(key):
    if key[0] == "gelu16":
        return "gemm_gelu16"
    if key[0] == "ln_mlp":
        return f"ln_mlp<{'true' if key[1] else 'false'}>"
    bn, amn, bmn, epi, ws = key
    return f"<{bn},{int(amn)},{int(bmn)},{epi},{int(ws)}>"


# ------------------------------------------------------------------------------------------ input families
FAMILIES = ("randn", "big", "small", "cancel", "exact")


def make_operands(family, M, N, K, seed, device, mn_major=False):
    """a, b (bf16, ops.gemm layout) of one family:
        randn      a ~ N(0, 1), b ~ N(0, 1) / sqrt(K)
        big, small randn times 2^20 / 2^-20 (a) and 2^10 / 2^-10 (b)
        cancel     every row of a is [v, -v] up to a small perturbation and b is [w, w]: sum a b ~ 0 while sum |a b|
                   is large, so only the budget's absolute part (kacc S) admits the result
        exact      integers in [-3, 3] (a) and [-2, 2] (b): every product and fp32 partial sum is exact"""
    g = torch.Generator(device="cpu").manual_seed(seed)
    if family == "exact":
        a = torch.randint(-3, 4, (M, K), generator=g).double()
        b = torch.randint(-2, 3, (N, K), generator=g).double()
    else:
        a = torch.randn(M, K, generator=g, dtype=torch.float64)
        b = torch.randn(N, K, generator=g, dtype=torch.float64) / math.sqrt(K)
        if family == "big":
            a, b = a * 2.0 ** 20, b * 2.0 ** 10
        elif family == "small":
            a, b = a * 2.0 ** -20, b * 2.0 ** -10
        elif family == "cancel":
            h = K // 2
            a[:, h:2 * h] = -a[:, :h] + 2.0 ** -6 * a[:, h:2 * h]
            b[:, h:2 * h] = b[:, :h]
        elif family != "randn":
            raise ValueError(family)
    a, b = a.bfloat16(), b.bfloat16()
    if mn_major:
        a, b = a.t(), b.t()
    return a.contiguous().to(device), b.contiguous().to(device)
