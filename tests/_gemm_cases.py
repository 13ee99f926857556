"""The GEMM variant matrix of tests/test_gemm_bounds_gpu.py as data (no GPU needed to list it): a covering list of
(shape, BN, operand majors, epilogue options, strides, input family) cases, with the kernel each one must reach at a
given SM count (tests/_gemm_ref.select_kernel).  tests/test_gemm_bounds_cpu.py checks that the list reaches every
kernel the built library contains."""
from __future__ import annotations

from dataclasses import dataclass

from tests import _gemm_ref as G

B200_SMS = 148


@dataclass(frozen=True)
class Case:
    M: int
    N: int
    K: int
    bn: int = 0
    mn: bool = False          # MN-major operands: wgrad, fp32 split-K reduce-add onto out
    splits: int = 1
    bias: bool = False
    res: str = ""             # "" | "res" | "inplace" (residual is out)
    out2: bool = False
    act: int = 0              # 0 | 1 GELU (aux_out unless noaux) | 2 GELU' (aux_in) | 3 ReLU
    noaux: bool = False
    colsum: bool = False
    dot: bool = False
    f32: bool = False
    drop: float = 0.0
    ln: str = ""              # "" | "skip" | "noskip": the LayerNorm-backward epilogue
    pad: int = 0              # extra columns of every leading dimension (lda, ldb, ldo, ldr, ld_aux, ld_dot)
    family: str = "randn"

    def kernel(self, sms=B200_SMS):
        return G.select_kernel(self.M, self.N, self.K, sms, bn=self.bn, mn_major=self.mn, splits=self.splits,
                               out_mode=2 if self.mn else (1 if self.f32 else 0), act=self.act,
                               residual=bool(self.res), dot=self.dot, drop=self.drop > 0, ln=bool(self.ln),
                               colsum=self.colsum)

    @property
    def id(self):
        opts = [k for k in ("mn", "bias", "out2", "noaux", "colsum", "dot", "f32") if getattr(self, k)]
        opts += [f"{k}{getattr(self, k)}" for k in ("res", "ln") if getattr(self, k)]
        opts += [f"act{self.act}"] if self.act else []
        opts += [f"splits{self.splits}"] if self.splits > 1 else []
        opts += [f"drop{self.drop}"] if self.drop else []
        opts += [f"pad{self.pad}"] if self.pad else []
        return f"{self.M}x{self.N}x{self.K}-bn{self.bn}-{'-'.join(opts) or 'plain'}-{self.family}"


EDGE_M = (1, 31, 32, 33, 127, 128, 129, 257)
EDGE_N = (8, 24, 56, 72, 120, 136, 200, 248, 264, 520)
EDGE_K = (8, 24, 56, 64, 72, 200, 256, 264, 592, 1536)
FAMS = ("randn", "exact", "cancel", "big", "small")
WS_M = 2 * B200_SMS * 128 + 1          # ragged, past 2 x 148 tiles of one n tile: weight-stationary
MANY_M = 4993                          # 40 m tiles: several items per CTA, both accumulator buffers


def _streaming():
    """Every streaming epilogue at every BN, over the edge shapes (each variant sees a rotation of M, N, K)."""
    opts = {
        0: [dict(), dict(bias=True), dict(bias=True, res="res"), dict(res="inplace", bias=True),
            dict(res="res", out2=True), dict(bias=True, colsum=True), dict(colsum=True), dict(dot=True),
            dict(act=3, bias=True), dict(bias=True, res="res", pad=8)],
        1: [dict(bias=True), dict(bias=True, noaux=True), dict(bias=True, colsum=True), dict(pad=16, bias=True)],
        2: [dict(), dict(colsum=True), dict(pad=8)],
        3: [dict(f32=True), dict(f32=True, bias=True), dict(f32=True, bias=True, pad=8)],
        6: [dict(act=1, bias=True, drop=0.1), dict(act=1, bias=True, noaux=True, drop=0.25)],
        7: [dict(res="res", bias=True, drop=0.1), dict(res="res", bias=True, out2=True, drop=0.3)],
    }
    out = []
    for bi, bn in enumerate((64, 128, 256)):
        for epi, lst in opts.items():
            for i, o in enumerate(lst):
                o = dict(o)
                if epi == 1:
                    o["act"] = 1
                if epi == 2:
                    o["act"] = 2
                j = 3 * i + 5 * bi + epi
                M, N, K = EDGE_M[j % len(EDGE_M)], EDGE_N[(j * 3 + 1) % len(EDGE_N)], EDGE_K[(j * 7 + 2) % len(EDGE_K)]
                if o.get("dot"):
                    N = (64, 128, 192, 512)[j % 4]
                fam = FAMS[j % len(FAMS)]
                if o.get("act") in (1,) or o.get("drop"):
                    fam = ("randn", "cancel", "small")[j % 3]
                out.append(Case(M, N, K, bn=bn, family=fam, **o))
    return out


def _many_items():
    return [Case(MANY_M, 520, 200, bn=64, bias=True, colsum=True), Case(MANY_M, 248, 72, bn=128, res="res", bias=True),
            Case(MANY_M, 264, 264, bn=256, act=1, bias=True), Case(MANY_M, 512, 64, bn=128, dot=True),
            Case(MANY_M, 136, 56, bn=128, act=2, colsum=True, family="exact"),
            Case(MANY_M, 120, 24, bn=64, f32=True, bias=True, family="exact")]


def _weight_stationary():
    out = []
    for bn in (128, 256):
        for K in (8, 56, 200, 256):
            out += [Case(WS_M, 256, K, bn=bn, bias=True, family="exact" if K == 56 else "randn"),
                    Case(WS_M, 256, K, bn=bn, f32=True, bias=True),
                    Case(WS_M, 256, K, bn=bn, colsum=True, bias=True) if K == 200 else
                    Case(WS_M, 256, K, bn=bn, act=3, bias=True, pad=8)]
        out += [Case(WS_M, 264 if bn == 128 else 512, 200, bn=bn, act=1, bias=True, colsum=True),   # generic GELU, WS
                Case(WS_M, 256, 72, bn=bn, act=1, bias=True, noaux=True, colsum=True)]
    # the 16-warp GELU kernel: N % 256 == 0, K <= 256, with and without aux_out
    out += [Case(WS_M, 256, 256, bn=256, act=1, bias=True), Case(WS_M, 512, 200, bn=0, act=1, bias=True, noaux=True),
            Case(WS_M, 256, 8, bn=256, act=1, bias=True, family="cancel")]
    # K = 264: one k-block past the resident slice, streams
    out += [Case(WS_M, 256, 264, bn=256, bias=True)]
    return out


def _wgrad():
    out = []
    for bn in (64, 128, 256):
        out += [Case(2560, 256, 200, bn=bn, mn=True, splits=4, family="exact"),
                Case(264, 72 if bn == 64 else 264, 1000, bn=bn, mn=True, splits=64, pad=8),   # splits past the k-blocks
                Case(40, 520, 129, bn=bn, mn=True, splits=3, family="cancel")]      # (MN-major: M is the row pitch)
    return out


def _ln_bwd():
    return [Case(M, 256, K, ln=ln, family=fam) for M, K, ln, fam in
            ((1, 256, "skip", "randn"), (33, 768, "noskip", "randn"), (129, 1024, "skip", "cancel"),
             (WS_M, 1024, "skip", "randn"), (MANY_M, 64, "noskip", "randn"), (257, 8, "skip", "randn"))]


CASES = _streaming() + _many_items() + _weight_stationary() + _wgrad() + _ln_bwd()


def model_cases():
    """nn.Linear forward / dgrad / wgrad shapes of the cfg 2 VTMAE at the benchmark batch (256) and of DinoV2
    (dinov2_vits14_reg) fine-tuning at B = 64, 224 x 224, derived from the module configurations."""
    from oracle.vtmae_oracle import VTMAEConfig
    cfg = VTMAEConfig()
    B = 256
    n_tok = cfg.n_img + cfg.num_tactiles * cfg.n_tac
    n_vis = n_tok - int(cfg.masking_ratio * n_tok)
    out = []
    for rows, dim, inner, mlp in ((B * n_vis, cfg.dim, cfg.heads * cfg.dim_head, cfg.mlp_dim),
                                  (B * n_tok, cfg.decoder_dim, cfg.decoder_heads * cfg.decoder_dim_head,
                                   4 * cfg.decoder_dim)):
        out += linear_shapes(rows, dim, inner, mlp)
    import inspect
    from m3l_b200.dinov2 import DinoV2
    d = {k: v.default for k, v in inspect.signature(DinoV2.__init__).parameters.items() if k != "self"}
    D, ps, B2 = d["embed_dim"], d["patch_size"], 64
    rows = B2 * (1 + d["num_register_tokens"] + (224 // ps) ** 2)
    out += linear_shapes(rows, D, D, d["mlp_ratio"] * D)
    P = 3 * ps * ps
    out.append(Case(B2 * (224 // ps) ** 2, D, (P + 7) // 8 * 8, bias=True))     # patch embedding, K padded to 8
    return out


def linear_shapes(R, dim, inner, mlp):
    """One transformer layer's products at R token rows: forward, dgrad (with the fused epilogues the engine uses) and
    wgrad (split-K over the rows, engine._wgrad_tiling)."""
    cs = [Case(R, 3 * inner, dim), Case(R, dim, inner, bias=True, res="res"),
          Case(R, mlp, dim, bias=True, act=1), Case(R, dim, mlp, bias=True, res="res"),
          Case(R, inner, dim, dot=True), Case(R, mlp, dim, act=2, colsum=True),
          Case(R, dim, 3 * inner) if dim != 256 else Case(R, dim, 3 * inner, ln="skip"),
          Case(R, dim, mlp, ln="skip") if dim == 256 else Case(R, dim, mlp)]
    for n_out, n_in in ((3 * inner, dim), (dim, inner), (mlp, dim), (dim, mlp)):
        bn, splits = _wgrad_tiling_static(n_out, n_in, R)
        cs.append(Case(n_out, n_in, R, bn=bn, mn=True, splits=splits))
    return cs


def _wgrad_tiling_static(n_out, n_in, rows, sms=B200_SMS):
    """engine._wgrad_tiling (which reads the SM count of the current device) at a given SM count."""
    bn = 256 if n_in % 256 == 0 else (128 if n_in % 128 == 0 else 64)
    tiles = ((n_out + 127) // 128) * ((n_in + bn - 1) // bn)
    kb = (rows + 63) // 64
    return bn, max(1, min(max(1, sms // tiles), kb))


# ln_mlp_fwd: (rows, hidden, output mode, save, family); modes: "new" (out = fresh buffer), "inplace" (out = x),
# "has_x" (out holds a copy of x)
LN_MLP = [(M, hidden, mode, save, fam) for (M, hidden), (mode, save), fam in zip(
    [(1, 128), (33, 512), (129, 1024), (WS_M + 4, 1024), (1, 1024), (33, 128), (129, 512), (257, 256), (MANY_M, 384)],
    [("new", False), ("inplace", False), ("has_x", True), ("inplace", True), ("has_x", False), ("has_x", True),
     ("new", False), ("inplace", True), ("has_x", True)],
    ["randn", "smallvar", "offset", "randn", "offset", "smallvar", "randn", "smallvar", "randn"])]
