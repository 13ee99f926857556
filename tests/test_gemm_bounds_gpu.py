"""GPU: every tcgen05 GEMM variant (csrc/gemm.cu, csrc/gemm_gelu.cu) and the fused feed-forward block (csrc/rowblock.cu)
element by element against the float64 reference of tests/_gemm_ref.py, within error budgets derived from where the
kernels round, at the tile edges of every variant (tests/_gemm_cases.py) and at the model shapes; that each case
reaches the kernel the host selection is meant to pick; that nothing is written outside the outputs, every output
element is written and nothing outside the operands is read; and the properties of the persistent schedule: two runs
and every row-prefix of A give bit-identical rows, a row of A reaches only its row of the output and a row of B only
its column.

M3L_GEMM_BOUNDS_REPORT=<path> writes the largest |err| / budget per (variant, output) there as JSON, with the name of
the device and whether the BN / weight-stationary variants of one product agreed bit for bit."""
import json
import math
import os
import zlib

import pytest
import torch

from tests import _dropout_ref as DR
from tests import _gemm_cases as K
from tests import _gemm_ref as G

pytestmark = pytest.mark.gpu

DEV = "cuda"
RATIOS = {}
BITWISE = {}
PAD_ROWS = 5
SENT16 = 0x7FA5                   # NaN bit patterns no kernel produces: surroundings of every output
SENT32 = 0x7FA5A5A5
DROP_KEY = 0x5DEECE66D


@pytest.fixture(scope="module")
def ops():
    from m3l_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("M3L_GEMM_BOUNDS_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump({"device": torch.cuda.get_device_name(0), "worst_ratio": {k: RATIOS[k] for k in sorted(RATIOS)},
                       "variants_bitwise_equal": BITWISE}, f, indent=1)


# ------------------------------------------------------------------------------------------ buffers
class Framed:
    """A [rows, cols] view (leading dimension ld) inside a larger buffer: PAD_ROWS rows before and after and columns
    cols..ld hold a sentinel bit pattern; the view itself is prefilled with `fill` (NaN for outputs)."""

    def __init__(self, rows, cols, ld, dtype, fill=math.nan):
        self.buf = torch.empty(rows + 2 * PAD_ROWS, ld, dtype=dtype, device=DEV)
        self.bits().fill_(SENT16 if dtype == torch.bfloat16 else SENT32)
        self.view = self.buf[PAD_ROWS:PAD_ROWS + rows, :cols]
        if isinstance(fill, torch.Tensor):
            self.view.copy_(fill)
        else:
            self.view.fill_(fill)
        self.mask = torch.ones(self.buf.shape, dtype=torch.bool, device=DEV)
        self.mask[PAD_ROWS:PAD_ROWS + rows, :cols] = False

    def bits(self):
        return self.buf.view(torch.int16 if self.buf.dtype == torch.bfloat16 else torch.int32)

    def check(self, name):
        sent = SENT16 if self.buf.dtype == torch.bfloat16 else SENT32
        outside = self.bits()[self.mask]
        bad = int((outside != sent).sum())
        assert bad == 0, f"{name}: {bad} elements written outside the output"
        unwritten = int((~torch.isfinite(self.view)).sum())
        assert unwritten == 0, f"{name}: {unwritten} output elements not written (or not finite)"


def poisoned(x, pad):
    """x [rows, cols] as a view with leading dimension cols + pad inside a buffer with 8 more rows; every element
    outside x is NaN, so a read past the operand's bounds shows in the result."""
    rows, cols = x.shape
    buf = torch.full((rows + 8, cols + pad), math.nan, dtype=x.dtype, device=DEV)
    buf[:rows, :cols] = x
    return buf[:rows, :cols]


def vec_framed(n, init):
    """An fp32 vector of n entries (initial values `init`) followed and preceded by sentinels."""
    f = Framed(1, n, n + 24, torch.float32, fill=init.view(1, n))
    return f


def launched(fn):
    """Run fn under the profiler; returns (result, [parsed kernel keys of the GEMM / ln_mlp launches])."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    keys = [k for k in map(G.parse_kernel_name, names) if k is not None]
    return res, keys if keys else names


def record(variant, name, r):
    key = f"{variant}/{name}"
    RATIOS[key] = max(RATIOS.get(key, 0.0), r)


# ------------------------------------------------------------------------------------------ one case
def side_inputs(c, seed):
    g = torch.Generator(device="cpu").manual_seed(seed + 1)
    M, N = c.M, c.N
    exact = c.family == "exact"
    ints = lambda *s, lo=-8, hi=9: torch.randint(lo, hi, s, generator=g).double()
    if exact:
        bias = ints(N).float()
        res = ints(M, N).bfloat16()
        aux = (torch.randint(-2, 3, (M, N), generator=g).double() / 2).bfloat16()
        init = ints(M, N).float() if c.mn else None
        cs0 = ints(N).float()
        side = ints(M, N, lo=-2, hi=3).bfloat16()
    else:
        sc = {"big": 2.0 ** 20, "small": 2.0 ** -20}.get(c.family, 1.0)
        bias = (torch.randn(N, generator=g, dtype=torch.float64) * sc).float()
        res = (torch.randn(M, N, generator=g, dtype=torch.float64) * sc).bfloat16()
        aux = (torch.rand(M, N, generator=g, dtype=torch.float64) * 1.2 - 0.1).bfloat16()
        init = (torch.randn(M, N, generator=g, dtype=torch.float64) * sc).float() if c.mn else None
        cs0 = torch.randn(N, generator=g, dtype=torch.float64).float()
        side = torch.randn(M, N, generator=g, dtype=torch.float64).bfloat16()
    to = lambda t: t.to(DEV) if t is not None else None
    return to(bias), to(res), to(aux), to(init), to(cs0), to(side)


def ln_inputs(c, seed):
    g = torch.Generator(device="cpu").manual_seed(seed + 2)
    x = torch.randn(c.M, 256, generator=g, dtype=torch.float64)
    mean = x.mean(1, keepdim=True)
    rstd = 1 / torch.sqrt(x.var(1, unbiased=False, keepdim=True) + 1e-5)
    stats = torch.cat([mean, rstd], 1).float()
    gamma = (torch.rand(256, generator=g, dtype=torch.float64) + 0.5).float()
    skip = torch.randn(c.M, 256, generator=g, dtype=torch.float64).bfloat16() if c.ln == "skip" else None
    inits = {k: torch.randn(256, generator=g, dtype=torch.float64).float().to(DEV)
             for k in ("dgamma", "dbeta", "dx_colsum")}
    return x.bfloat16().to(DEV), stats.to(DEV), gamma.to(DEV), (skip.to(DEV) if skip is not None else None), inits


def run_case(ops, c, seed):
    """Calls the kernel on framed / poisoned buffers.  Returns (dict of outputs, dict of Framed, inputs)."""
    a, b = G.make_operands(c.family, c.M, c.N, c.K, seed, DEV, mn_major=c.mn)
    A, B = poisoned(a, c.pad), poisoned(b, c.pad)
    bias, res, aux, init, cs0, side = side_inputs(c, seed)
    M, N, ld = c.M, c.N, c.N + c.pad
    fr, kw = {}, {}
    if c.ln:
        x, stats, gamma, skip, inits = ln_inputs(c, seed)
        fr["out"] = Framed(M, N, N, torch.bfloat16)
        for k, v in inits.items():
            fr[k] = vec_framed(N, v)
        kw["ln_bwd"] = dict(x=x, stats=stats, gamma=gamma, skip=skip, dgamma=fr["dgamma"].view.view(-1),
                            dbeta=fr["dbeta"].view.view(-1), dx_colsum=fr["dx_colsum"].view.view(-1))
        inputs = dict(a=a, b=b, x=x, stats=stats, gamma=gamma, skip=skip, inits=inits)
        ops.gemm(A, B, out=fr["out"].view, **kw)
        return {k: (f.view if k == "out" else f.view.view(-1)) for k, f in fr.items()}, fr, inputs
    if c.mn:
        fr["out"] = Framed(M, N, ld, torch.float32, fill=init)
        kw.update(mn_major=True, accumulate=True, splits=c.splits)
    elif c.res == "inplace":
        fr["out"] = Framed(M, N, ld, torch.bfloat16, fill=res)
        kw["residual"] = fr["out"].view
    else:
        fr["out"] = Framed(M, N, ld, torch.float32 if c.f32 else torch.bfloat16)
        if c.res:
            kw["residual"] = poisoned(res, c.pad)
    if c.bias:
        kw["bias"] = bias
    if c.out2:
        fr["out2"] = Framed(M, N, ld, torch.bfloat16)
        kw["out2"] = fr["out2"].view
    if c.act:
        kw["act"] = c.act
    if c.act == 1 and not c.noaux:
        fr["aux"] = Framed(M, N, ld, torch.bfloat16)
        kw["aux_out"] = fr["aux"].view
    if c.act == 2:
        kw["aux_in"] = poisoned(aux, c.pad)
    if c.colsum:
        fr["colsum"] = vec_framed(N, cs0)
        kw["colsum_out"] = fr["colsum"].view.view(-1)
    if c.dot:
        fr["dot"] = Framed(M, N // 64, N // 64, torch.float32)
        kw["dot_side"] = poisoned(side, c.pad)
        kw["dot_out"] = fr["dot"].view
    if c.drop:
        key = torch.tensor([DROP_KEY], dtype=torch.int64, device=DEV)
        kw["dropout"] = ops.Dropout(key, 6 if c.act == 1 else 7, c.drop)
    ops.gemm(A, B, out=fr["out"].view, bn=c.bn, **kw)
    outs = {k: (f.view.view(-1) if k == "colsum" else f.view) for k, f in fr.items()}
    inputs = dict(a=a, b=b, bias=bias if c.bias else None, res=res if c.res else None, aux=aux, init=init, cs0=cs0,
                  side=side)
    return outs, fr, inputs


def reference(c, outs, inp):
    """{name: (want, budget, exact)} for every output of the case."""
    if c.ln:
        r = G.ln_bwd_reference(inp["a"], inp["b"], inp["x"], inp["stats"], inp["gamma"], inp["skip"], inp["inits"])
        return {k: (r.want[k], r.budget[k], False) for k in ("dx", "dgamma", "dbeta", "dx_colsum")}
    keep = None
    if c.drop:
        keep = torch.from_numpy(DR.mask(DROP_KEY, 6 if c.act == 1 else 7, c.M, c.N, c.drop)).to(DEV)
    r = G.gemm_reference(inp["a"], inp["b"], mn_major=c.mn, bias=inp["bias"], residual=inp["res"], act=c.act,
                         aux_in=inp["aux"] if c.act == 2 else None, out_f32=c.f32,
                         init=inp["init"] if c.mn else None, splits=G.clamp_splits(c.K, c.splits), keep=keep,
                         exact=c.family == "exact")
    ref = {"out": (r.want["out"], r.budget["out"], "out" in r.exact)}
    if "out2" in outs:
        ref["out2"] = ref["out"]
    if "aux" in outs:
        ref["aux"] = (r.want["aux"], r.budget["aux"], False)
    if "dot" in outs:
        w, e = G.rowdot_reference(outs["out"], inp["side"])
        ref["dot"] = (w, e, False)
    if "colsum" in outs:
        w, e = G.colsum_reference(outs["out"], inp["cs0"])
        ref["colsum"] = (w, e, False)
    return ref, keep


def check_case(ops, c, seed, sms):
    (outs, fr, inp), keys = launched(lambda: run_case(ops, c, seed))
    want_key = c.kernel(sms)
    assert keys == [want_key], f"{c.id}: launched {[G.variant_label(k) for k in keys]}, the host selection mirror " \
                               f"expects {G.variant_label(want_key)}"
    for name, f in fr.items():
        f.check(f"{c.id} {name}")
    ref = reference(c, outs, inp)
    ref, keep = ref if isinstance(ref, tuple) else (ref, None)
    failures = []
    label = G.variant_label(want_key)
    for name, (want, budget, exact) in ref.items():
        got = outs["out" if name == "dx" else name]
        if exact:
            w = want.float().to(got.dtype)
            if not torch.equal(got, w):
                bad = torch.nonzero(got != w)[0].tolist()
                failures.append(f"{name}: exact family, not bit-identical at {bad}: got {float(got[tuple(bad)])}, "
                                f"want {float(w[tuple(bad)])}")
        if keep is not None and name in ("out", "aux", "out2") and c.act == 1:
            dropped = keep == 0
            if not (got[dropped] == 0).all():
                failures.append(f"{name}: dropped elements not exactly 0")
        g2, w2, b2 = (got, want, budget) if got.dim() == 2 else (got[None], want[None], budget[None])
        r, msg = G.ratio(name, g2, w2, b2)
        record(label, name, r)
        if not r <= 1.0:
            failures.append(msg)
    assert not failures, f"{c.id} ({label})\n" + "\n".join(failures)
    return outs


# ------------------------------------------------------------------------------------------ ln_mlp_fwd
def ln_mlp_inputs(M, hidden, family, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(M, 256, generator=g, dtype=torch.float64)
    if family == "smallvar":
        x = x * 0.03
    elif family == "offset":
        x = 4 + 0.05 * x
    w1 = torch.randn(hidden, 256, generator=g, dtype=torch.float64) / 16
    w2 = torch.randn(256, hidden, generator=g, dtype=torch.float64) / math.sqrt(hidden)
    gamma = torch.rand(256, generator=g, dtype=torch.float64) + 0.5
    beta = torch.randn(256, generator=g, dtype=torch.float64) * 0.1
    b1 = torch.randn(hidden, generator=g, dtype=torch.float64) * 0.1
    b2 = torch.randn(256, generator=g, dtype=torch.float64) * 0.1
    bf = lambda t: t.bfloat16().to(DEV).contiguous()
    f32 = lambda t: t.float().to(DEV)
    return bf(x), f32(gamma), f32(beta), bf(w1), f32(b1), bf(w2), f32(b2)


@pytest.mark.parametrize("M,hidden,mode,save,family", K.LN_MLP)
def test_ln_mlp_within_budget(ops, M, hidden, mode, save, family):
    """The fused feed-forward block in its three output modes, its training outputs (stats, xn, h, gp) each against
    their own budget, sentinels around every output."""
    x, gamma, beta, w1, b1, w2, b2 = ln_mlp_inputs(M, hidden, family, seed=M + hidden)
    x0 = x.clone()
    fo = Framed(M, 256, 256, torch.bfloat16, fill=x if mode != "new" else math.nan)
    kw = {}
    if save:
        fr = dict(stats=Framed(M, 2, 2, torch.float32), xn=Framed(M, 256, 256, torch.bfloat16),
                  h=Framed(M, hidden, hidden, torch.bfloat16), gp=Framed(M, hidden, hidden, torch.bfloat16))
    else:
        fr = {}
    if mode == "inplace":
        xin, kw["out"] = fo.view, fo.view
        assert fo.view.is_contiguous()
    else:
        xin, kw["out"] = x, fo.view
        kw["out_has_x"] = mode == "has_x"

    def call():
        if not save:
            return ops.ln_mlp_fwd(xin, gamma, beta, w1, b1, w2, b2, **kw)
        # the wrapper allocates the training outputs; copy them into framed buffers via a second, framed call
        from m3l_b200 import _lib
        import ctypes as C
        a = _lib.LnMlpArgs()
        a.x, a.rows, a.dim, a.hidden = _lib.ptr(xin), M, 256, hidden
        a.gamma, a.beta, a.eps = _lib.ptr(gamma), _lib.ptr(beta), 1e-5
        a.w1, a.b1, a.w2, a.b2 = _lib.ptr(w1), _lib.ptr(b1), _lib.ptr(w2), _lib.ptr(b2)
        a.out, a.out_has_x = _lib.ptr(fo.view), int(mode == "has_x")
        a.stats, a.xn_out, a.h_out, a.gp_out = (_lib.ptr(fr[k].view) for k in ("stats", "xn", "h", "gp"))
        _lib.check(_lib.load().m3l_ln_mlp_fwd(C.byref(a), _lib.current_stream()), "m3l_ln_mlp_fwd")

    _, keys = launched(call)
    assert keys == [("ln_mlp", save)], keys
    fo.check("out")
    for k, f in fr.items():
        f.check(k)
    saved = (fr["stats"].view, fr["xn"].view, fr["h"].view, fr["gp"].view) if save else None
    r = G.ln_mlp_reference(x0, gamma, beta, w1, b1, w2, b2, 1e-5, saved=saved, two_roundings=mode != "new")
    got = {"out": fo.view}
    if save:
        got.update(mean=fr["stats"].view[:, 0:1], rstd=fr["stats"].view[:, 1:2], xn=fr["xn"].view, h=fr["h"].view,
                   gp=fr["gp"].view)
    failures = []
    for name, g in got.items():
        rr, msg = G.ratio(name, g, r.want[name], r.budget[name])
        record(f"ln_mlp<{'true' if save else 'false'}>", name, rr)
        if not rr <= 1.0:
            failures.append(msg)
    assert not failures, f"M={M} hidden={hidden} mode={mode} save={save} {family}\n" + "\n".join(failures)


# ------------------------------------------------------------------------------------------ the variant matrix
@pytest.mark.parametrize("c", K.CASES, ids=lambda c: c.id)
def test_variant_matrix_within_budget(ops, sms, c):
    check_case(ops, c, seed=zlib.crc32(c.id.encode()) % 10007, sms=sms)


@pytest.mark.parametrize("c", K.model_cases(), ids=lambda c: c.id)
def test_model_shapes_within_budget(ops, sms, c):
    check_case(ops, c, seed=7, sms=sms)


def test_repeat_runs_are_bit_identical(ops, sms):
    """Two identical calls give identical outputs (the fp32 atomics and split-K reduce-adds are checked against their
    budgets in the matrix instead)."""
    for c in [x for x in K.CASES if not x.mn and not x.ln][::3]:
        o1, _, _ = run_case(ops, c, 3)
        o2, _, _ = run_case(ops, c, 3)
        for name in o1:
            if name not in ("colsum",):
                assert torch.equal(o1[name], o2[name]), f"{c.id}: {name} differs between two identical calls"


# ------------------------------------------------------------------------------------------ schedule properties
PREFIX = [(1000, 136, 200, 64), (1000, 264, 72, 128), (1000, 512, 264, 256), (K.WS_M + 300, 256, 200, 256)]


@pytest.mark.parametrize("M,N,Kd,bn", PREFIX)
def test_row_prefix_is_bit_identical(ops, sms, M, N, Kd, bn):
    """gemm(A[:M']) equals the first M' rows of gemm(A) for M' across tile and lane-quadrant edges, within one
    variant: a row's output does not depend on M, on the other rows or on which CTA / accumulator buffer ran it."""
    a, b = G.make_operands("randn", M, N, Kd, 5, DEV)
    bias = torch.randn(N, device=DEV)
    full = ops.gemm(a, b, bias=bias, bn=bn)
    key = G.select_kernel(M, N, Kd, sms, bn=bn)
    primes = (1, 31, 32, 33, 127, 128, 129, 257, 300) if key[4] is False else (K.WS_M - 4, K.WS_M + 1, M - 1)
    for m in primes:
        assert G.select_kernel(m, N, Kd, sms, bn=bn) == key
        part = ops.gemm(a[:m], b, bias=bias, bn=bn)
        assert torch.equal(part, full[:m]), f"M'={m}: rows differ from the M={M} run ({G.variant_label(key)})"


@pytest.mark.parametrize("M,N,Kd,bn,dot", [(700, 520, 200, 64, False), (700, 512, 264, 128, True),
                                           (K.WS_M, 256, 256, 256, False), (700, 256, 1536, 256, True)])
def test_rows_and_columns_are_isolated(ops, M, N, Kd, bn, dot):
    """Changing row i of A changes only row i of out (and of dot_out); changing row j of B changes only column j (and
    only dot group j // 64)."""
    a, b = G.make_operands("randn", M, N, Kd, 6, DEV)
    side = torch.randn(M, N, device=DEV).bfloat16()

    def run(a_, b_):
        if dot:
            d = torch.empty(M, N // 64, device=DEV)
            return ops.gemm(a_, b_, bn=bn, dot_side=side, dot_out=d), d
        return ops.gemm(a_, b_, bn=bn), None

    o0, d0 = run(a, b)
    for i in (0, 31, 32, 127, 128, M - 1):
        a2 = a.clone()
        a2[i] = torch.randn(Kd, device=DEV).bfloat16()
        o1, d1 = run(a2, b)
        rows = torch.nonzero((o1 != o0).any(1)).flatten().tolist()
        assert rows == [i], f"row {i} of A changed rows {rows[:8]}"
        if dot:
            assert torch.nonzero((d1 != d0).any(1)).flatten().tolist() == [i]
    for j in (0, 63, 64, N - 1):
        b2 = b.clone()
        b2[j] = torch.randn(Kd, device=DEV).bfloat16()
        o1, d1 = run(a, b2)
        cols = torch.nonzero((o1 != o0).any(0)).flatten().tolist()
        assert cols == [j], f"row {j} of B changed columns {cols[:8]}"
        if dot:
            assert torch.nonzero((d1 != d0).any(0)).flatten().tolist() == [j // 64]


@pytest.mark.parametrize("M,N,Kd,act", [(1000, 512, 200, 0), (1000, 512, 256, 1), (K.WS_M, 256, 200, 0),
                                        (K.WS_M, 256, 256, 1), (1000, 256, 1536, 2)])
def test_variants_agree_within_budget(ops, sms, M, N, Kd, act):
    """The same product through BN 64 / 128 / 256 (and, at WS_M rows, the weight-stationary and streaming kernels, by
    way of BN 64, which never runs weight-stationary): each within its budget; bitwise agreement is recorded."""
    a, b = G.make_operands("randn", M, N, Kd, 8, DEV)
    bias = torch.randn(N, device=DEV) if act != 2 else None
    aux = (torch.rand(M, N, device=DEV) * 1.2 - 0.1).bfloat16() if act == 2 else None
    r = G.gemm_reference(a, b, bias=bias, act=act, aux_in=aux)
    outs = {}
    for bn in (64, 128, 256):
        key = G.select_kernel(M, N, Kd, sms, bn=bn, act=act)
        o = ops.gemm(a, b, bn=bn, bias=bias, act=act, aux_in=aux)
        rr, msg = G.ratio("out", o, r.want["out"], r.budget["out"])
        record(G.variant_label(key), "out", rr)
        assert rr <= 1.0, f"bn={bn} ({G.variant_label(key)}): {msg}"
        outs[G.variant_label(key)] = o
    labels = list(outs)
    BITWISE[f"{M}x{N}x{Kd} act{act}"] = {f"{x} == {y}": bool(torch.equal(outs[x], outs[y]))
                                         for i, x in enumerate(labels) for y in labels[i + 1:]}
