"""GPU: the attention kernels element by element against the float64 reference of tests/_attn_ref.py, within error
budgets derived from where the kernels round, at every sequence length of the n <= 256 kernels (csrc/attention.cu)
and on input families that hide masking and rounding errors from random data; and the properties of their persistent
schedules: bit-identical results for every batch size and run, no influence between (sample, head) items, no write
outside the outputs and no element left unwritten.  The 32- / 128-wide and n > 256 kernels (attention_dh.cu,
attention_long.cu) get the same checks through mha_fwd / mha_bwd.

M3L_ATTN_BOUNDS_REPORT=<path> writes the largest |err| / budget per kernel family and output there as JSON."""
import json
import math
import os

import pytest
import torch

from tests import _attn_ref as R

pytestmark = pytest.mark.gpu

DEV = "cuda"
RATIOS = {}


@pytest.fixture(scope="module")
def ops():
    from m3l_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("M3L_ATTN_BOUNDS_REPORT")
    if path:
        with open(path, "w") as f:
            json.dump({k: RATIOS[k] for k in sorted(RATIOS)}, f, indent=1)


def kernel_family(n, dh):
    if dh != 64:
        return f"dh{dh}"
    return "small" if n <= 16 else "tcgen05" if n <= 256 else "long"


def kernels(ops, n, dh):
    """attention_fwd / _bwd where they apply (the kernels under test), mha_fwd / _bwd (which selects) elsewhere."""
    if not R.is_long(n, dh):
        return ops.attention_fwd, ops.attention_bwd
    return ops.mha_fwd, ops.mha_bwd


def delta_of(out, dout, B, n, H, dh):
    """rowsum(dout * out) per (token, head) in fp32 from the bf16 out: what engine.py passes the backward."""
    return (dout.float() * out.float()).view(B * n, H, dh).sum(-1).contiguous()


def grads(dqkv, B, n, H, dh):
    dq, dk, dv = dqkv.view(B, n, 3, H, dh).permute(2, 0, 3, 1, 4)
    return dict(dq=dq, dk=dk, dv=dv)


def check_budgets(ops, qkv, dout, B, n, H, dh, scale):
    fwd, bwd = kernels(ops, n, dh)
    out, lse = fwd(qkv, B, n, H, dh, scale)
    ref = R.reference(qkv, dout, B, n, H, dh, scale, out=out, lse=lse)
    got = [("", "out", R.heads_view(out, B, n, H, dh)), ("", "lse", lse)]
    for mode, d in (("delta=None", None), ("delta given", delta_of(out, dout, B, n, H, dh))):
        dqkv = bwd(qkv, out, dout, lse, B, n, H, dh, scale, delta=d)
        got += [(mode, k, v) for k, v in grads(dqkv, B, n, H, dh).items()]
    fam = kernel_family(n, dh)
    failures = []
    for mode, name, g in got:
        r, msg = R.worst_ratio(name, g, getattr(ref, name), ref.budget[name])
        RATIOS[f"{fam}/{name}"] = max(RATIOS.get(f"{fam}/{name}", 0.0), r)
        if not r <= 1.0:
            failures.append(f"{msg} [{mode}]" if mode else msg)
    assert not failures, f"B={B} n={n} H={H} dh={dh} scale={scale:g}\n" + "\n".join(failures)


# ------------------------------------------------------------------------------------------ budgets
@pytest.mark.parametrize("n", range(1, 257))
def test_every_length_within_budget(ops, n):
    """Every n of the short kernels: the n <= 16 / tcgen05 switch, NK = round_up(n, 16), the 64-key P slabs, the
    query rows split over two tiles above 128, the backward's 64-row second tile (129..192) and its buffering (193)."""
    B, H = 3, 2
    qkv, dout = R.make_inputs("randn", B, n, H, 64, 0.125, seed=n, device=DEV)
    check_budgets(ops, qkv, dout, B, n, H, 64, 0.125)


EDGE_N = [1, 10, 16, 17, 64, 65, 128, 129, 192, 193, 255, 256]
CASES = [(f, 64 ** -0.5) for f in R.FAMILIES] + [("randn", 1.0), ("randn", 0.01)]


@pytest.mark.parametrize("family,scale", CASES)
@pytest.mark.parametrize("n", EDGE_N)
def test_input_families_within_budget(ops, family, scale, n):
    B, H = 2, 2
    qkv, dout = R.make_inputs(family, B, n, H, 64, scale, seed=100 + n, device=DEV)
    check_budgets(ops, qkv, dout, B, n, H, 64, scale)


@pytest.mark.parametrize("n", [17, 192])
def test_sixteen_heads_within_budget(ops, n):
    """H = 16: qkv rows 3072 wide."""
    B, H = 2, 16
    qkv, dout = R.make_inputs("randn", B, n, H, 64, 0.125, seed=7, device=DEV)
    check_budgets(ops, qkv, dout, B, n, H, 64, 0.125)


OTHER = [(dh, n) for dh in (32, 128) for n in (1, 17, 129, 256, 257, 385)] + [(64, 257), (64, 385)]


@pytest.mark.parametrize("family,scale", CASES)
@pytest.mark.parametrize("dh,n", OTHER)
def test_other_kernels_within_budget(ops, family, scale, dh, n):
    """attention_dh (32- and 128-wide heads) and attention_long (n > 256); dominant_last puts the largest score of every
    row in the last key tile, so the online softmax rescales its accumulator there."""
    B, H = 2, 2
    scale = scale * math.sqrt(64 / dh)
    qkv, dout = R.make_inputs(family, B, n, H, dh, scale, seed=200 + n, device=DEV)
    check_budgets(ops, qkv, dout, B, n, H, dh, scale)


# ------------------------------------------------------------------------------------------ schedule properties
def run_all(ops, qkv, dout, B, n, H, dh, scale):
    """out, lse, dqkv (delta=None), dqkv (delta given)."""
    fwd, bwd = kernels(ops, n, dh)
    out, lse = fwd(qkv, B, n, H, dh, scale)
    d0 = bwd(qkv, out, dout, lse, B, n, H, dh, scale)
    d1 = bwd(qkv, out, dout, lse, B, n, H, dh, scale, delta=delta_of(out, dout, B, n, H, dh))
    return out, lse, d0, d1


def per_sample(x, B):
    """[B*n, ...] or [B, ...] -> B slices"""
    return x.view(B, -1)


NAMES = ("out", "lse", "dqkv (delta=None)", "dqkv (delta given)")
# (dh, B, n, H).  tcgen05: B*H >= 3 * 148 SMs and not a multiple of it, so every CTA runs several items and both ring
# slots; n <= 16: B*H > 8 * 148 * 4 warps, so warps loop; the benchmark's decoder (n = 192) and encoder (n = 10)
MANY_ITEMS = [(64, 256, 192, 4), (64, 256, 10, 4), (64, 113, 129, 4), (64, 113, 192, 4), (64, 113, 193, 4),
              (64, 113, 256, 4), (64, 1200, 10, 4), (64, 40, 385, 4), (32, 40, 257, 4), (128, 40, 129, 4)]


@pytest.mark.parametrize("dh,B,n,H", MANY_ITEMS)
def test_batch_invariant_and_deterministic(ops, dh, B, n, H):
    """Each (sample, head) item is computed the same whichever CTA / warp / ring slot runs it and whatever ran before
    it: two runs are bit-identical, and so is every sample to a B = 1 run of it alone."""
    scale = dh ** -0.5
    qkv, dout = R.make_inputs("randn", B, n, H, dh, scale, seed=11, device=DEV)
    first = run_all(ops, qkv, dout, B, n, H, dh, scale)
    second = run_all(ops, qkv, dout, B, n, H, dh, scale)
    for name, a, b in zip(NAMES, first, second):
        assert torch.equal(a, b), f"{name} differs between two identical runs"
    full = [per_sample(t, B) for t in first]
    for b in range(B):
        rows = slice(b * n, (b + 1) * n)
        alone = run_all(ops, qkv[rows].contiguous(), dout[rows].contiguous(), 1, n, H, dh, scale)
        for name, f, a in zip(NAMES, full, alone):
            assert torch.equal(f[b], a.view(-1)), f"sample {b}: {name} differs from a B = 1 run of it"


ISOLATION = [(64, 1200, 10, 4), (64, 113, 129, 4), (64, 113, 192, 4), (64, 113, 256, 4), (64, 40, 385, 4),
             (32, 40, 257, 4), (128, 40, 129, 4)]


@pytest.mark.parametrize("poison", [math.nan, math.inf])
@pytest.mark.parametrize("dh,B,n,H", ISOLATION)
def test_items_are_isolated(ops, poison, dh, B, n, H):
    """One sample's qkv and dout are NaN / Inf: every other sample's out, lse and dqkv are bit-identical to a clean run.
    A value left over from a previous item and masked by multiplying (0 * NaN = NaN) instead of selecting shows here."""
    scale = dh ** -0.5
    qkv, dout = R.make_inputs("randn", B, n, H, dh, scale, seed=12, device=DEV)
    bad = 5                       # its items' CTAs (tcgen05: items 20..23 of 452) run clean items next
    rows = slice(bad * n, (bad + 1) * n)
    qkv_p, dout_p = qkv.clone(), dout.clone()
    qkv_p[rows] = poison
    dout_p[rows] = poison
    clean = [per_sample(t, B) for t in run_all(ops, qkv, dout, B, n, H, dh, scale)]
    dirty = [per_sample(t, B) for t in run_all(ops, qkv_p, dout_p, B, n, H, dh, scale)]
    keep = torch.arange(B, device=DEV) != bad
    for name, c, d in zip(NAMES, clean, dirty):
        assert torch.equal(c[keep], d[keep]), \
            f"{name}: samples {sorted(set(torch.nonzero((c != d).any(1) & keep).flatten().tolist()))} changed"


BOUNDS = [(64, n) for n in (1, 10, 16, 17, 128, 129, 192, 193, 256, 385)] + [(32, 129), (128, 257)]
SENTINEL = -1024.0               # exact in bf16 and fp32


def nan_prefix_buffer(numel, dtype, extra=1024):
    """A buffer of numel NaN followed by `extra` sentinels; returns (buffer, prefix view)."""
    buf = torch.full((numel + extra,), SENTINEL, dtype=dtype, device=DEV)
    buf[:numel] = math.nan
    return buf, buf[:numel]


def nan_tailed_copy(x, extra=1024):
    """x as the prefix of a larger buffer whose tail is NaN: a read past x that is masked by multiplying yields NaN."""
    buf = torch.full((x.numel() + extra,), math.nan, dtype=x.dtype, device=DEV)
    buf[:x.numel()] = x.flatten()
    return buf[:x.numel()].view(x.shape)


@pytest.mark.parametrize("dh,n", BOUNDS)
def test_outputs_written_exactly_within_their_buffers(ops, dh, n):
    """Outputs prefilled with NaN inside larger sentinel-filled buffers: every element is written (finite), nothing past
    the end is; lse and delta given as prefixes of NaN-filled buffers; the results equal those of plain buffers."""
    B, H = 3, 2
    inner, scale = H * dh, dh ** -0.5
    fwd, bwd = kernels(ops, n, dh)
    qkv, dout = R.make_inputs("randn", B, n, H, dh, scale, seed=13, device=DEV)
    out_ref, lse_ref, d0_ref, d1_ref = run_all(ops, qkv, dout, B, n, H, dh, scale)
    out_buf, out_v = nan_prefix_buffer(B * n * inner, torch.bfloat16)
    lse_buf, lse_v = nan_prefix_buffer(B * H * n, torch.float32)
    out, lse = fwd(qkv, B, n, H, dh, scale, out=out_v.view(B * n, inner), lse=lse_v.view(B, H, n))
    for name, buf, v, ref in (("out", out_buf, out_v, out_ref), ("lse", lse_buf, lse_v, lse_ref)):
        assert (buf[v.numel():] == SENTINEL).all(), f"{name}: written past its end"
        assert torch.isfinite(v).all(), f"{name}: {int((~torch.isfinite(v)).sum())} elements not written"
        assert torch.equal(v, ref.flatten()), f"{name} differs from a run with plain buffers"
    delta = delta_of(out, dout, B, n, H, dh)
    for name, d, ref in (("delta=None", None, d0_ref), ("delta given", nan_tailed_copy(delta), d1_ref)):
        dq_buf, dq_v = nan_prefix_buffer(B * n * 3 * inner, torch.bfloat16)
        bwd(qkv, out, dout, nan_tailed_copy(lse), B, n, H, dh, scale, dqkv=dq_v.view(B * n, 3 * inner), delta=d)
        assert (dq_buf[dq_v.numel():] == SENTINEL).all(), f"dqkv ({name}): written past its end"
        assert torch.isfinite(dq_v).all(), f"dqkv ({name}): {int((~torch.isfinite(dq_v)).sum())} elements not finite"
        assert torch.equal(dq_v, ref.flatten()), f"dqkv ({name}) differs from a run with plain buffers"


ENTRY = {"small": "m3l_attention", "tcgen05": "m3l_attention", "long": "m3l_attention_long",
         "dh32": "m3l_attention_dh", "dh128": "m3l_attention_dh"}


@pytest.mark.parametrize("dh,n", [(64, 10), (64, 192), (64, 385), (32, 129), (128, 257)])
def test_empty_batch_touches_nothing(dh, n):
    """batch = 0 returns success and writes nothing.  The C entry points are called directly with pointers to real
    buffers: they reject null pointers before they look at the batch, and torch gives an empty tensor a null one."""
    import ctypes as C
    from m3l_b200 import _lib
    lib = _lib.load()
    entry = ENTRY[kernel_family(n, dh)]
    H, scale = 2, C.c_float(dh ** -0.5)
    inner = H * dh
    qkv = torch.randn(n, 3 * inner, device=DEV).bfloat16()
    dout = torch.randn(n, inner, device=DEV).bfloat16()
    lse_in = torch.zeros(H * n, device=DEV)
    delta = torch.zeros(n, H, device=DEV)
    out_buf = torch.full((n * inner,), SENTINEL, device=DEV).bfloat16()
    lse_buf = torch.full((H * n,), SENTINEL, device=DEV)
    dq_buf = torch.full((n * 3 * inner,), SENTINEL, device=DEV).bfloat16()
    p, stream = _lib.ptr, _lib.current_stream()
    _lib.check(getattr(lib, entry + "_fwd")(p(qkv), 0, n, H, dh, scale, p(out_buf), p(lse_buf), stream), entry)
    for d in (None, delta):
        _lib.check(getattr(lib, entry + "_bwd")(p(qkv), p(out_buf), p(dout), p(lse_in), p(d), 0, n, H, dh, scale,
                                                  p(dq_buf), stream), entry)
    torch.cuda.synchronize()
    for name, buf in (("out", out_buf), ("lse", lse_buf), ("dqkv", dq_buf)):
        assert (buf == SENTINEL).all(), f"{name}: written with batch = 0"
