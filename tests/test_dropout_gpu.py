"""GPU: dropout in training mode.  The kernels' masks are bit-exact against the numpy definition (tests/_dropout_ref.py);
at p = 0 the dropout kernels are bit-identical to the kernels without dropout; attention with dropout matches a float64
reference that uses the numpy mask; every module that runs the transformer stack matches the oracle with the same
masks; CUDA graphs, seeds and eval mode behave as nn.Dropout users expect."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import vtmae_oracle as O
from tests import _dropout_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel_err(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / (b.abs().max() + 1e-30)).item()


def cos(a, b):
    a, b = a.double().flatten().cpu(), b.double().flatten().cpu()
    return float(a @ b / (a.norm() * b.norm() + 1e-300))


@pytest.fixture(scope="module")
def ops():
    from m3l_b200 import ops as _ops
    return _ops


def _key(k):
    return torch.tensor([k], dtype=torch.int64, device=DEV)


# ---------------------------------------------------------------------------------------------- masks
@pytest.mark.parametrize("rows,cols,key,site,p", [
    (300, 256, 0x0123456789ABCDEF, 5, 0.1), (70000, 13, 7, 3, 0.5), (129, 1000, (1 << 62) - 1, 1023, 0.25),
    (1, 8, 0, 0, 0.9), (4096, 24, 0x5555AAAA5555, 14, 0.5)])
def test_masks_are_bit_exact(ops, rows, cols, key, site, p):
    ones = torch.ones(rows, cols, dtype=torch.bfloat16, device=DEV)
    colsum = torch.zeros(cols, dtype=torch.float32, device=DEV)
    z = ops.dropout_bwd(ones, ops.Dropout(_key(key), site, p), colsum=colsum)
    ref = R.mask(key, site, rows, cols, p)
    zb = torch.from_numpy(ref).to(torch.bfloat16)
    assert torch.equal(z.cpu(), zb)
    assert torch.allclose(colsum.cpu(), zb.float().sum(0), rtol=1e-5, atol=1e-3)


# ---------------------------------------------------------------------------------------------- attention
_NS = [1, 10, 17, 128, 129, 256, 257, 1374]
_DHS = [32, 64, 128]


def _plain(ops, dh):
    return (ops.attention_long_fwd, ops.attention_long_bwd) if dh == 64 else (ops.attention_dh_fwd, ops.attention_dh_bwd)


def _case(B, n, H, dh, seed=3):
    g = torch.Generator(device=DEV).manual_seed(seed)
    qkv = torch.randn(B * n, 3 * H * dh, device=DEV, generator=g).bfloat16()
    dout = torch.randn(B * n, H * dh, device=DEV, generator=g).bfloat16()
    return qkv, dout


@pytest.mark.parametrize("dh", _DHS)
@pytest.mark.parametrize("n", _NS)
def test_attention_dropout_at_p0_is_bit_identical(ops, dh, n):
    B, H = 2, 2
    qkv, dout = _case(B, n, H, dh)
    scale = dh ** -0.5
    fwd, bwd = _plain(ops, dh)
    o0, l0 = fwd(qkv, B, n, H, dh, scale)
    d = ops.Dropout(_key(12345), 4, 0.0)
    o1, l1 = ops.attention_dropout_fwd(qkv, B, n, H, dh, scale, d)
    assert torch.equal(o0, o1) and torch.equal(l0, l1)
    delta = (dout.float() * o0.float()).reshape(B * n, H, dh).sum(-1).contiguous()
    for dl in (None, delta):
        assert torch.equal(bwd(qkv, o0, dout, l0, B, n, H, dh, scale, delta=dl),
                           ops.attention_dropout_bwd(qkv, o0, dout, l0, B, n, H, dh, scale, d, delta=dl))


def _ref64(qkv, dout, B, n, H, dh, scale, z):
    qr = qkv.double().requires_grad_(True)
    q, k, v = qr.reshape(B, n, 3, H, dh).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-1, -2)) * scale
    o = ((torch.softmax(s, -1) * z) @ v).transpose(1, 2).reshape(B * n, H * dh)
    o.backward(dout.double())
    return o.detach(), torch.logsumexp(s, -1).detach(), qr.grad


@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("dh", _DHS)
@pytest.mark.parametrize("n", _NS)
def test_attention_dropout_vs_float64(ops, p, dh, n):
    B, H = 2, 2
    key, site = 0x1234_5678_9ABC + n, (3 << 2) | 0
    qkv, dout = _case(B, n, H, dh, seed=n)
    scale = dh ** -0.5
    d = ops.Dropout(_key(key), site, p)
    out, lse = ops.attention_dropout_fwd(qkv, B, n, H, dh, scale, d)
    z = torch.from_numpy(R.attn_mask(key, site, B, H, n, p)).to(DEV, torch.float64)
    oref, lref, gref = _ref64(qkv, dout, B, n, H, dh, scale, z)
    assert torch.isfinite(out.float()).all()
    assert rel_err(out, oref) < 2e-2
    _, l0 = _plain(ops, dh)[0](qkv, B, n, H, dh, scale)
    assert torch.equal(lse, l0)                       # lse of the undropped scores
    assert (lse.double() - lref).abs().max().item() < 2e-2
    inner = H * dh
    delta = (dout.float() * out.float()).reshape(B * n, H, dh).sum(-1).contiguous()
    for dl in (None, delta):
        dqkv = ops.attention_dropout_bwd(qkv, out, dout, lse, B, n, H, dh, scale, d, delta=dl)
        for name, sl in (("dq", slice(0, inner)), ("dk", slice(inner, 2 * inner)), ("dv", slice(2 * inner, 3 * inner))):
            if n == 1 and name != "dv":
                # one key: dS = P (Z dP - delta) is exactly 0, the kernel leaves the rounding of delta, which comes from
                # the bf16 output Z v (Z = 65536 / (65536 - thr) makes that rounding nonzero)
                assert dqkv[:, sl].float().abs().max() < 1e-2 * gref.abs().max(), name
                continue
            assert cos(dqkv[:, sl], gref[:, sl]) > 0.999, (name, dl is None)
            assert rel_err(dqkv[:, sl], gref[:, sl]) < 5e-2, (name, dl is None)
    # same key: bit-identical; another key: another output (from 10 tokens on: with one key per row, both masks
    # often keep all four rows)
    out2, _ = ops.attention_dropout_fwd(qkv, B, n, H, dh, scale, d)
    assert torch.equal(out, out2)
    assert torch.equal(dqkv, ops.attention_dropout_bwd(qkv, out, dout, lse, B, n, H, dh, scale, d, delta=delta))
    if n >= 10:
        out3, _ = ops.attention_dropout_fwd(qkv, B, n, H, dh, scale, ops.Dropout(_key(key + 1), site, p))
        assert not torch.equal(out, out3)


def test_mha_routes_dropout(ops):
    B, n, H, dh = 2, 10, 4, 64
    qkv, _ = _case(B, n, H, dh)
    d = ops.Dropout(_key(5), 0, 0.3)
    assert torch.equal(ops.mha_fwd(qkv, B, n, H, dh, 0.125, dropout=d)[0],
                       ops.attention_dropout_fwd(qkv, B, n, H, dh, 0.125, d)[0])


def test_opcheck_dropout_ops():
    import m3l_b200.torch_ops  # noqa: F401
    B, n, H, dh = 2, 130, 2, 32
    qkv, dout = _case(B, n, H, dh)
    key = _key(77)
    OPS = torch.ops.m3l
    torch.library.opcheck(OPS.attention_dropout_fwd, (qkv, B, n, H, dh, dh ** -0.5, key, 2, 0.2))
    o, lse = OPS.attention_dropout_fwd(qkv, B, n, H, dh, dh ** -0.5, key, 2, 0.2)
    torch.library.opcheck(OPS.attention_dropout_bwd, (qkv, o, dout, lse, B, n, H, dh, dh ** -0.5, key, 2, 0.2))
    torch.library.opcheck(OPS.dropout_bwd, (dout, key, 3, 0.2))


# ---------------------------------------------------------------------------------------------- GEMM epilogues
@pytest.mark.parametrize("M,K,N", [(2560, 256, 512), (1000, 256, 256), (300, 512, 256)])
def test_gemm_dropout_epilogues(ops, M, K, N):
    g = torch.Generator(device=DEV).manual_seed(M)
    a = (torch.randn(M, K, device=DEV, generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, device=DEV, generator=g) * 0.05).bfloat16()
    bias = torch.randn(N, device=DEV, generator=g) * 0.1
    res = torch.randn(M, N, device=DEV, generator=g).bfloat16()
    key = _key(0xABCDEF)
    # p = 0: bit-identical to the plain epilogues
    pre0, pre1 = torch.empty(M, N, dtype=torch.bfloat16, device=DEV), torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
    h0 = ops.gemm(a, w, bias=bias, act=ops.GELU_FWD, aux_out=pre0)
    h1 = ops.gemm(a, w, bias=bias, act=ops.GELU_FWD, aux_out=pre1, dropout=ops.Dropout(key, 6, 0.0))
    assert torch.equal(h0, h1) and torch.equal(pre0, pre1)
    o0 = ops.gemm(a, w, bias=bias, residual=res)
    o1 = ops.gemm(a, w, bias=bias, residual=res, dropout=ops.Dropout(key, 7, 0.0))
    assert torch.equal(o0, o1)
    # p > 0: the numpy mask applied to the fp32 epilogue values
    p = 0.1
    acc = a.float() @ w.float().T + bias
    z2 = torch.from_numpy(R.mask(0xABCDEF, 6, M, N, p)).to(DEV)
    z3 = torch.from_numpy(R.mask(0xABCDEF, 7, M, N, p)).to(DEV)
    h = ops.gemm(a, w, bias=bias, act=ops.GELU_FWD, aux_out=pre1, dropout=ops.Dropout(key, 6, p))
    gelu = torch.nn.functional.gelu(acc)
    assert torch.equal(h == 0, (z2 == 0) | (h0 == 0))
    assert rel_err(h.float(), gelu * z2) < 1e-2
    gp = 0.5 * (1 + torch.erf(acc / 2 ** 0.5)) + acc * torch.exp(-0.5 * acc * acc) / (2 * np.pi) ** 0.5
    assert rel_err(pre1.float(), gp * z2) < 1e-2
    out2 = torch.empty(M, N, dtype=torch.bfloat16, device=DEV)
    o = ops.gemm(a, w, bias=bias, residual=res, out2=out2, dropout=ops.Dropout(key, 7, p))
    assert torch.equal(o, out2)
    assert rel_err(o.float(), res.float() + z3 * acc) < 1e-2


# ---------------------------------------------------------------------------------------------- modules
_KEY_TENSORS = {}


@contextlib.contextmanager
def known_keys(keys):
    """engine.draw_dropout_key hands out these keys, cycling in call order."""
    from m3l_b200 import engine
    # kept for the life of the process: captured CUDA graphs read the keys from these addresses
    dev_keys = _KEY_TENSORS.setdefault(tuple(keys), torch.tensor(keys, dtype=torch.int64, device=DEV))
    state = {"i": 0}

    def draw(device):
        i = state["i"] % len(keys)
        state["i"] += 1
        return dev_keys[i:i + 1]

    orig = engine.draw_dropout_key
    engine.draw_dropout_key = draw
    try:
        yield state
    finally:
        engine.draw_dropout_key = orig


def _build(cfg, sd, p):
    from m3l_b200 import VTT, VTMAE
    enc = VTT(image_size=cfg.image_size, tactile_size=cfg.tactile_size, image_patch_size=cfg.image_patch_size,
              tactile_patch_size=cfg.tactile_patch_size, dim=cfg.dim, depth=cfg.depth, heads=cfg.heads,
              mlp_dim=cfg.mlp_dim, image_channels=cfg.image_channels, tactile_channels=cfg.tactile_channels,
              dim_head=cfg.dim_head, num_tactiles=cfg.num_tactiles, frame_stack=cfg.frame_stack, dropout=p)
    mae = VTMAE(encoder=enc, decoder_dim=cfg.decoder_dim, masking_ratio=cfg.masking_ratio,
                decoder_depth=cfg.decoder_depth, decoder_heads=cfg.decoder_heads,
                decoder_dim_head=cfg.decoder_dim_head, num_tactiles=cfg.num_tactiles,
                early_conv_masking=cfg.early_conv_masking, use_sincosmod_encodings=cfg.use_sincosmod_encodings,
                frame_stack=cfg.frame_stack)
    mae.load_state_dict(O.expand_aliases({k: v.detach().clone() for k, v in sd.items()}), strict=True)
    return mae.to(DEV)


def _inputs(cfg, B, seed):
    gen = torch.Generator().manual_seed(seed)
    H, W = cfg.image_size
    th, tw = cfg.tactile_size
    x = {"image": torch.rand(B, 3 * cfg.frame_stack, H, W, generator=gen),
         "tactile1": torch.rand(B, 3 * cfg.frame_stack, th, tw, generator=gen),
         "tactile2": torch.rand(B, 3 * cfg.frame_stack, th, tw, generator=gen)}
    noise = O.tie_free_noise(B, cfg.n_img + 2 * cfg.n_tac, gen, [cfg.n_img, cfg.n_tac, cfg.n_tac])
    return x, noise


def _to_dev(x):
    return {k: v.to(DEV) for k, v in x.items()}


def _check_grads(named, sd, keys, tol=0.999):
    for k in keys:
        gr = sd[k].grad
        if gr is None or float(gr.abs().max()) == 0.0:
            assert named[k].grad is None or float(named[k].grad.abs().max()) == 0.0, k
            continue
        assert cos(named[k].grad, gr) >= tol, (k, cos(named[k].grad, gr))


@pytest.mark.parametrize("dh,heads", [(64, 4), (32, 8), (128, 2)])
def test_transformer_dropout_vs_oracle(dh, heads):
    from m3l_b200.vtmae import Transformer
    torch.manual_seed(5)
    dim, depth, mlp, p, B, n = 256, 2, 512, 0.2, 3, 40
    t = Transformer(dim, depth, heads, dh, mlp, dropout=p)
    sd = {"t." + k: v.detach().clone().requires_grad_(True) for k, v in t.state_dict().items()}
    t = t.to(DEV).train()
    x = torch.randn(B, n, dim)
    xd = x.to(DEV).requires_grad_(True)
    key = 0x0BADC0FFEE
    with known_keys([key]):
        y = t(xd)
    xr = x.double().requires_grad_(True)
    yr = R.transformer(xr, {k: v.double() for k, v in sd.items()}, "t", depth, heads, dh, drop=R.MaskHook(key, p))
    assert cos(y, yr.detach()) >= 0.9995
    w = torch.randn(B, n, dim)
    (y * w.to(DEV)).sum().backward()
    (yr * w.double()).sum().backward()
    assert cos(xd.grad, xr.grad) >= 0.999
    named = {"t." + k: v for k, v in t.named_parameters()}
    _check_grads(named, sd, list(sd))


def test_vtmae_dropout_loss_gradients_and_embeddings_vs_oracle():
    cfg = O.VTMAEConfig(depth=2, decoder_depth=2)
    sd = O.init_state_dict(cfg, seed=2)
    x, noise = _inputs(cfg, 4, 3)
    p = 0.1
    mae = _build(cfg, sd, p)
    mae.use_cuda_graph = False
    mae.train()
    key = 0x1111_2222_3333
    with known_keys([key]):
        loss = mae(_to_dev(x), noise=noise.to(DEV))
    loss.backward()
    for k in O.param_keys(sd):
        sd[k].requires_grad_(True)
    with R.oracle_dropout({"encoder.transformer": R.MaskHook(key, p)}):
        lref = O.vtmae_forward(sd, cfg, x, noise)
    lref.backward()
    assert abs(loss.item() - lref.item()) <= 1e-2 * abs(lref.item()), (loss.item(), lref.item())
    _check_grads(dict(mae.named_parameters(remove_duplicate=False)), sd, O.param_keys(sd))
    # get_embeddings in training mode (eval=False), all tokens
    with known_keys([key + 1]), torch.no_grad():
        emb = mae.get_embeddings(_to_dev(x), eval=False)
    with R.oracle_dropout({"encoder.transformer": R.MaskHook(key + 1, p)}), torch.no_grad():
        eref = O.vtmae_embeddings({k: v.detach() for k, v in sd.items()}, cfg, x)
    assert cos(emb, eref) >= 0.9995


def test_mae_extractor_dropout_vs_oracle():
    """MAEExtractor with dropout in the MAE encoder (p_mae) and in the extra block (p_vit): forward under no_grad
    and with the gradients into both."""
    from m3l_b200 import MAEExtractor
    cfg = O.VTMAEConfig(depth=2)
    sd = O.init_state_dict(cfg, seed=4)
    gen = torch.Generator().manual_seed(6)
    B, F_ = 3, cfg.frame_stack
    obs = {"image": torch.rand(B, F_, 64, 64, 3, generator=gen),
           "tactile": torch.rand(B, F_, 6, 32, 32, generator=gen) * 2 - 1}
    p_mae, p_vit = 0.1, 0.2
    mae = _build(cfg, sd, p_mae)
    torch.manual_seed(9)
    ext = MAEExtractor(None, mae, cfg.dim, False, F_).to(DEV)
    ext.vit_layer.transformer.p_drop = p_vit
    ext.use_cuda_graph = False
    sd_vit = {"transformer." + k: v.detach().cpu().clone() for k, v in ext.vit_layer.transformer.state_dict().items()}
    k1, k2 = 0x77, 0x78
    hooks = {"encoder.transformer": R.MaskHook(k1, p_mae), "transformer": R.MaskHook(k2, p_vit)}
    with known_keys([k1, k2]), torch.no_grad():
        f0 = ext({k: v.clone().to(DEV) for k, v in obs.items()})
    with R.oracle_dropout(hooks), torch.no_grad():
        r0 = O.extractor_forward(sd, cfg, sd_vit, {k: v.clone() for k, v in obs.items()})
    assert cos(f0, r0) >= 0.9995
    w = torch.randn(B, cfg.dim, generator=gen)
    with known_keys([k1, k2]):
        feats = ext({k: v.clone().to(DEV) for k, v in obs.items()})
    assert torch.equal(feats.detach(), f0)
    (feats * w.to(DEV)).sum().backward()
    for k in O.param_keys(sd):
        sd[k].requires_grad_(True)
    for v in sd_vit.values():
        v.requires_grad_(True)
    with R.oracle_dropout(hooks):
        ref = O.extractor_forward(sd, cfg, sd_vit, {k: v.clone() for k, v in obs.items()})
    (ref * w).sum().backward()
    for k, prm in ext.vit_layer.transformer.named_parameters():
        assert cos(prm.grad, sd_vit["transformer." + k].grad) >= 0.999, k
    _check_grads(dict(mae.named_parameters(remove_duplicate=False)), sd, O.param_keys(sd))


def test_joint_pass_dropout_vs_oracle():
    """The joint MAE + extractor pass (one embedding of all tokens, graph-replayed) with encoder dropout: loss against
    the oracle's masked pass and features against the oracle's extractor, with the masks of the keys the pass drew
    (all-token encoder, then masked encoder; the extra block has no dropout here)."""
    from m3l_b200 import MAEExtractor
    cfg = O.VTMAEConfig(depth=2, decoder_depth=2)
    sd = O.init_state_dict(cfg, seed=8)
    gen = torch.Generator().manual_seed(21)
    B, p = 6, 0.1
    mae = _build(cfg, sd, p)
    ext = MAEExtractor(None, mae, cfg.dim, False, cfg.frame_stack).to(DEV)
    sd_vit = {"transformer." + k: v.detach().cpu().clone() for k, v in ext.vit_layer.transformer.state_dict().items()}
    obs = {"image": torch.rand(B, cfg.frame_stack, 64, 64, 3, generator=gen),
           "tactile": torch.rand(B, cfg.frame_stack, 6, 32, 32, generator=gen) * 2 - 1}
    noise = O.tie_free_noise(B, 192, gen, [64] * 3)
    kA, kB = 101, 202
    with R.oracle_dropout({"encoder.transformer": R.MaskHook(kA, p)}), torch.no_grad():
        fref = O.extractor_forward(sd, cfg, sd_vit, {k: v.clone() for k, v in obs.items()})
    for rep in range(2):                 # graph capture, replay (the keys are fixed at capture)
        ext.zero_grad(set_to_none=True)
        with known_keys([kA, kB]):
            l_j = ext.joint_mae_loss({k: v.to(DEV) for k, v in obs.items()}, noise=noise.to(DEV))
        f_j = ext({k: v.to(DEV) for k, v in obs.items()})
        assert cos(f_j.detach(), fref) >= 0.9995, rep
        ((f_j ** 2).sum() + l_j).backward()
        if rep == 0:
            l0 = l_j.detach().clone()
        else:
            assert torch.equal(l_j.detach(), l0)
    xs = _maps_from_obs(obs, cfg)
    with R.oracle_dropout({"encoder.transformer": R.MaskHook(kB, p)}), torch.no_grad():
        lref = O.vtmae_forward({k: v.detach() for k, v in sd.items()}, cfg, xs, noise)
    assert abs(l0.item() - lref.item()) <= 1e-2 * abs(lref.item()), (l0.item(), lref.item())


def _maps_from_obs(obs, cfg):
    """The oracle's vt_load of raw 5-D observations, as MAEExtractor feeds the MAE."""
    o = dict(obs)
    im = o["image"].permute(0, 2, 3, 1, 4)
    o["image"] = im.reshape(im.shape[0], im.shape[1], im.shape[2], -1)
    t = o["tactile"]
    o["tactile"] = t.reshape(t.shape[0], -1, t.shape[3], t.shape[4])
    return O.vt_load(o, frame_stack=cfg.frame_stack)


def test_vtt_dino_dropout_with_masks_and_registers_vs_oracle():
    from oracle import vtt_dino_oracle as VD
    from m3l_b200.vtt import VTT
    cfg = VD.VTTDinoConfig(image_size=(64, 64), tactile_size=(64, 64), image_patch_size=8, tactile_patch_size=8, depth=2,
                           num_register_tokens=2)
    torch.manual_seed(21)
    p = 0.15
    m = VTT(image_size=cfg.image_size, tactile_size=cfg.tactile_size, image_patch_size=cfg.image_patch_size,
            tactile_patch_size=cfg.tactile_patch_size, dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, mlp_dim=cfg.mlp_dim,
            num_tactiles=cfg.num_tactiles, image_channels=cfg.image_channels, tactile_channels=cfg.tactile_channels,
            dim_head=cfg.dim_head, num_register_tokens=cfg.num_register_tokens, pos_embed_fn="sinusoidal", dropout=p)
    with torch.no_grad():
        m.register_tokens.normal_(0, 0.5)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(DEV).train()
    g = torch.Generator().manual_seed(31)
    B = 2
    x = {"image": torch.rand(B, 12, 64, 64, generator=g), "tactile1": torch.rand(B, 12, 64, 64, generator=g),
         "tactile2": torch.rand(B, 12, 64, 64, generator=g)}
    masks = [torch.stack([torch.randperm(64, generator=g)[:40] for _ in range(B)]) for _ in range(2)]
    key = 0x4242
    with known_keys([key]):
        out = m.forward_features(_to_dev(x), [mk.to(DEV) for mk in masks])
    for k in sd:
        if sd[k].dtype.is_floating_point and k != "pos_embed.frequency_bands":
            sd[k].requires_grad_(True)
    with R.oracle_dropout({"transformer": R.MaskHook(key, p)}):
        ref = VD.forward_features(sd, cfg, x, masks)
    for k in ("x_norm_regtokens", "x_norm_patchtokens", "x_prenorm"):
        assert cos(out[k], ref[k].detach()) >= 0.9995, k
    w = torch.randn(ref["x_norm_patchtokens"].shape, generator=g)
    (out["x_norm_patchtokens"] * w.to(DEV)).sum().backward()
    (ref["x_norm_patchtokens"] * w).sum().backward()
    for k, prm in m.named_parameters():
        gr = sd[k].grad
        if gr is None or float(gr.abs().max()) == 0.0:
            continue
        assert prm.grad is not None and cos(prm.grad, gr) >= 0.999, k


def test_fused_train_steps_dropout_vs_oracle():
    """Three FusedTrainer steps (CUDA graph replays), each with its own known key, against the oracle's train_step
    with the same masks."""
    cfg = O.VTMAEConfig()
    sd = O.init_state_dict(cfg, seed=4)
    x, noise = _inputs(cfg, 8, 17)
    p = 0.1
    mae = _build(cfg, sd, p)
    mae.train()
    mae.initialize_training({"lr": 1e-4, "batch_size": 8})
    mae._trainer.use_graph = False
    st = O.AdamWState()
    xd, nd = _to_dev(x), noise.to(DEV)
    w0 = {k: v.detach().clone() for k, v in sd.items()}
    for it, key in enumerate([0x10, 0x20, 0x30]):
        with known_keys([key]):
            l = mae.train_step(xd, noise=nd)
        with R.oracle_dropout({"encoder.transformer": R.MaskHook(key, p)}):
            lo, norm, _ = O.train_step(sd, cfg, x, noise, st)
        assert abs(l.item() - lo.item()) <= 1e-2 * abs(lo.item()), (it, l.item(), lo.item())
        assert abs(mae._trainer.state[2].item() - norm.item()) <= 3e-2 * norm.item()
    named = dict(mae.named_parameters())
    for k in ["encoder.transformer.layers.0.0.to_qkv.weight", "encoder.transformer.layers.1.1.net.4.bias",
              "encoder.transformer.layers.0.0.to_out.0.bias", "decoder.layers.0.1.net.1.weight", "to_pixels.weight"]:
        upd_ref = sd[k].detach() - w0[k]
        upd = named[k].detach().cpu() - w0[k]
        assert cos(upd, upd_ref) >= 0.99, (k, cos(upd, upd_ref))


# ---------------------------------------------------------------------------------------------- graphs and seeds
def _vtmae_pair(p, seed=5):
    cfg = O.VTMAEConfig(depth=2, decoder_depth=1)
    sd = O.init_state_dict(cfg, seed=seed)
    x, noise = _inputs(cfg, 4, seed)
    return cfg, sd, _to_dev(x), noise.to(DEV)


def test_graph_path_equals_eager_and_replays_draw_fresh_masks():
    cfg, sd, x, noise = _vtmae_pair(0.1)
    mae_g, mae_e = _build(cfg, sd, 0.1), _build(cfg, sd, 0.1)
    mae_e.use_cuda_graph = False
    losses = []
    for it in range(3):
        torch.manual_seed(100 + it)
        lg = mae_g(x, noise=noise)
        lg.backward()
        torch.manual_seed(100 + it)
        le = mae_e(x, noise=noise)
        le.backward()
        if it > 0:                    # the first call captures (warm-up and capture draw keys too)
            assert torch.equal(lg.detach(), le.detach()), it
        losses.append(lg.item())
    # replays on the same inputs with fresh keys give different losses
    l1 = mae_g(x, noise=noise).item()
    l2 = mae_g(x, noise=noise).item()
    assert l1 != l2


def test_manual_seed_makes_eager_runs_bit_identical():
    cfg, sd, x, noise = _vtmae_pair(0.1, seed=6)
    mae = _build(cfg, sd, 0.1)
    mae.use_cuda_graph = False
    out = []
    for _ in range(2):
        torch.manual_seed(7)
        with torch.no_grad():
            out.append(mae.get_embeddings(x, eval=False))
    assert torch.equal(out[0], out[1])
    torch.manual_seed(8)
    with torch.no_grad():
        assert not torch.equal(mae.get_embeddings(x, eval=False), out[0])


def test_eval_mode_ignores_dropout():
    cfg, sd, x, noise = _vtmae_pair(0.1, seed=7)
    m1, m0 = _build(cfg, sd, 0.3), _build(cfg, sd, 0.0)
    for m in (m1, m0):
        m.eval()
    with torch.no_grad():
        assert torch.equal(m1(x, noise=noise), m0(x, noise=noise))
        assert torch.equal(m1.get_embeddings(x, eval=True), m0.get_embeddings(x, eval=True))
