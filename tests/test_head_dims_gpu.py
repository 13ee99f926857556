"""GPU: attention for 32- and 128-wide heads (csrc/attention_dh.cu) against a plain fp32 torch statement, and the
transformer modules built with those head widths against the oracle."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
DHS = (32, 128)


def rel_err(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


def cos(a, b):
    a, b = a.float().flatten(), b.float().flatten()
    return (a @ b / (a.norm() * b.norm() + 1e-30)).item()


@pytest.fixture(scope="module")
def ops():
    from m3l_b200 import ops as _ops
    return _ops


def _attn_ref(qkv, B, n, H, dh, scale):
    q, k, v = qkv.float().reshape(B, n, 3, H, dh).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-1, -2)) * scale
    return (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * n, H * dh), torch.logsumexp(s, -1)


def _check_vs_ref(ops, qkv, B, n, H, dh, seed=11):
    scale = dh ** -0.5
    out, lse = ops.attention_dh_fwd(qkv, B, n, H, dh, scale)
    qr = qkv.float().requires_grad_(True)
    oref, lref = _attn_ref(qr, B, n, H, dh, scale)
    assert torch.isfinite(out.float()).all() and torch.isfinite(lse).all()
    assert rel_err(out, oref) < 2e-2
    assert (lse - lref).abs().max().item() < 2e-2
    g = torch.Generator(device=DEV).manual_seed(seed)
    dout = torch.randn(B * n, H * dh, device=DEV, generator=g).bfloat16()
    oref.backward(dout.float())
    inner = H * dh
    delta = (dout.float() * out.float()).reshape(B * n, H, dh).sum(-1).contiguous()
    for d in (None, delta):
        dqkv = ops.attention_dh_bwd(qkv, out, dout, lse, B, n, H, dh, scale, delta=d)
        assert torch.isfinite(dqkv.float()).all()
        for name, sl in (("dq", slice(0, inner)), ("dk", slice(inner, 2 * inner)), ("dv", slice(2 * inner, 3 * inner))):
            if n == 1 and name != "dv":
                # one key: softmax is constant, dS and with it dQ and dK are exactly zero; the kernel leaves the bf16
                # rounding of dP - delta
                assert dqkv[:, sl].float().abs().max() < 1e-4 * qr.grad.abs().max(), (name, d is None)
                continue
            assert cos(dqkv[:, sl], qr.grad[:, sl]) > 0.999, (name, d is None)
            assert rel_err(dqkv[:, sl], qr.grad[:, sl]) < 5e-2, (name, d is None)


_SHAPES = [(3, 1, 2), (4, 10, 3), (2, 16, 2), (2, 17, 3), (2, 127, 2), (2, 128, 2), (2, 129, 3), (2, 192, 2),
           (2, 256, 2), (2, 257, 1), (2, 261, 3), (1, 384, 2), (1, 1000, 2), (1, 1374, 2), (1, 4096, 1),
           (64, 261, 4)]                 # 64 * 4 * 3 = 768 (sample, head, tile) items: more than SMs


@pytest.mark.parametrize("dh", DHS)
@pytest.mark.parametrize("B,n,H", _SHAPES)
def test_head_dim_attention_vs_fp32(ops, dh, B, n, H):
    torch.manual_seed(7)
    qkv = torch.randn(B * n, 3 * H * dh, device=DEV).bfloat16()
    _check_vs_ref(ops, qkv, B, n, H, dh)


@pytest.mark.parametrize("dh", DHS)
@pytest.mark.parametrize("B,n,H", [(2, 300, 2), (1, 1000, 3)])
def test_online_softmax_rescaling(ops, dh, B, n, H):
    """The largest score of many rows sits in the LAST key tile (spike keys along the direction every query leans
    to), so the running max grows late by more than the rescaling threshold and O must be rescaled."""
    torch.manual_seed(3)
    x = torch.randn(B, n, 3, H, dh, device=DEV)
    last0 = (n - 1) // 128 * 128
    spikes = torch.arange(last0, n, 7, device=DEV)
    u = torch.nn.functional.normalize(torch.randn(H, dh, device=DEV), dim=-1)
    # the spike keys are 40 u as at dh = 64 and the query lean grows with sqrt(dh): scaled spike scores of ~10, the
    # same jump as in the dh = 64 test
    x[:, :, 0] += 2.0 * (dh / 64) ** 0.5 * u
    x[:, spikes, 1] = 40.0 * u
    qkv = x.reshape(B * n, 3 * H * dh).bfloat16().contiguous()
    _check_vs_ref(ops, qkv, B, n, H, dh)


@pytest.mark.parametrize("dh", DHS)
@pytest.mark.parametrize("B,n,H", [(2, 1374, 3), (64, 261, 4)])
def test_head_dim_attention_is_deterministic(ops, dh, B, n, H):
    torch.manual_seed(9)
    scale = dh ** -0.5
    qkv = torch.randn(B * n, 3 * H * dh, device=DEV).bfloat16()
    dout = torch.randn(B * n, H * dh, device=DEV).bfloat16()
    runs = []
    for _ in range(2):
        o, l = ops.attention_dh_fwd(qkv, B, n, H, dh, scale)
        runs.append((o, l, ops.attention_dh_bwd(qkv, o, dout, l, B, n, H, dh, scale)))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("dh", DHS)
@pytest.mark.parametrize("n", [10, 261])
def test_no_writes_past_the_end(ops, dh, n):
    """Outputs are prefixes of larger sentinel-filled buffers: rows beyond B*n (and heads beyond H in lse) stay intact."""
    torch.manual_seed(4)
    B, H, scale, extra = 2, 3, dh ** -0.5, 200
    inner = H * dh
    qkv = torch.randn(B * n, 3 * inner, device=DEV).bfloat16()
    sentinel = -1234.0
    out_buf = torch.full(((B * n + extra) * inner,), sentinel, device=DEV).bfloat16()
    lse_buf = torch.full((B * H * n + extra,), sentinel, device=DEV)
    out = out_buf[:B * n * inner].view(B * n, inner)
    lse = lse_buf[:B * H * n].view(B, H, n)
    ops.attention_dh_fwd(qkv, B, n, H, dh, scale, out=out, lse=lse)
    assert (out_buf[B * n * inner:] == sentinel).all() and (lse_buf[B * H * n:] == sentinel).all()
    o_ref, l_ref = _attn_ref(qkv, B, n, H, dh, scale)
    assert rel_err(out, o_ref) < 2e-2 and (lse - l_ref).abs().max().item() < 2e-2
    dq_buf = torch.full(((B * n + extra) * 3 * inner,), sentinel, device=DEV).bfloat16()
    dqkv = dq_buf[:B * n * 3 * inner].view(B * n, 3 * inner)
    dout = torch.randn(B * n, inner, device=DEV).bfloat16()
    ops.attention_dh_bwd(qkv, out, dout, lse, B, n, H, dh, scale, dqkv=dqkv)
    assert (dq_buf[B * n * 3 * inner:] == sentinel).all()
    assert torch.isfinite(dqkv.float()).all()


@pytest.mark.parametrize("dh", DHS)
@pytest.mark.parametrize("n", [10, 256, 300])
def test_mha_sends_other_head_widths_to_the_new_kernels(ops, dh, n):
    torch.manual_seed(6)
    B, H, scale = 2, 2, dh ** -0.5
    qkv = torch.randn(B * n, 3 * H * dh, device=DEV).bfloat16()
    o, l = ops.mha_fwd(qkv, B, n, H, dh, scale)
    o_r, l_r = ops.attention_dh_fwd(qkv, B, n, H, dh, scale)
    assert torch.equal(o, o_r) and torch.equal(l, l_r)
    dout = torch.randn_like(o)
    assert torch.equal(ops.mha_bwd(qkv, o, dout, l, B, n, H, dh, scale),
                       ops.attention_dh_bwd(qkv, o, dout, l, B, n, H, dh, scale))


def test_errors_are_loud(ops):
    from m3l_b200._lib import M3LError
    qkv = torch.randn(2 * 30, 3 * 2 * 64, device=DEV).bfloat16()
    with pytest.raises(M3LError, match="status 3"):
        ops.attention_dh_fwd(qkv, 2, 30, 2, 64, 0.125)


@pytest.mark.parametrize("dh", DHS)
def test_opcheck_head_dim_attention(dh):
    import m3l_b200.torch_ops  # noqa: F401  (registers torch.ops.m3l)
    OPS = torch.ops.m3l
    torch.manual_seed(2)
    B, n, H = 2, 150, 2
    qkv = torch.randn(B * n, 3 * H * dh, device=DEV).bfloat16()
    torch.library.opcheck(OPS.attention_dh_fwd.default, (qkv, B, n, H, dh, dh ** -0.5))
    o, lse = OPS.attention_dh_fwd(qkv, B, n, H, dh, dh ** -0.5)
    torch.library.opcheck(OPS.attention_dh_bwd.default, (qkv, o, torch.randn_like(o), lse, B, n, H, dh, dh ** -0.5))


# ------------------------------------------------------------------------------ models
def _dcos(a, b):
    a, b = a.detach().double().flatten().cpu(), b.detach().double().flatten().cpu()
    return float(a @ b / (a.norm() * b.norm() + 1e-300))


def _to_dev(x):
    return {k: v.to(DEV) for k, v in x.items()}


# (encoder heads, encoder dim_head, decoder heads, decoder dim_head): inner = dim for the first; the second has
# encoder inner 64 and decoder inner 512 against dim 256
_VTMAE_CASES = [(8, 32, 2, 128), (2, 32, 4, 128)]


def _vtmae_case(heads, dh, dheads, ddh, B, seed):
    from oracle import vtmae_oracle as O
    cfg = O.VTMAEConfig(depth=2, decoder_depth=2, heads=heads, dim_head=dh, decoder_heads=dheads, decoder_dim_head=ddh)
    sd = O.init_state_dict(cfg, seed=seed)
    gen = torch.Generator().manual_seed(seed + 50)
    H, W = cfg.image_size
    th, tw = cfg.tactile_size
    x = {"image": torch.rand(B, 3 * cfg.frame_stack, H, W, generator=gen),
         "tactile1": torch.rand(B, 3 * cfg.frame_stack, th, tw, generator=gen),
         "tactile2": torch.rand(B, 3 * cfg.frame_stack, th, tw, generator=gen)}
    noise = O.tie_free_noise(B, cfg.n_img + 2 * cfg.n_tac, gen, [cfg.n_img, cfg.n_tac, cfg.n_tac])
    return cfg, sd, x, noise


@pytest.mark.parametrize("heads,dh,dheads,ddh", _VTMAE_CASES)
def test_vtmae_head_dims_vs_oracle(heads, dh, dheads, ddh):
    """Mask indices bit-exact, loss, every gradient, embeddings."""
    from oracle import vtmae_oracle as O
    from tests._build import build_product
    B = 4
    cfg, sd, x, noise = _vtmae_case(heads, dh, dheads, ddh, B, seed=1)
    mae = build_product(cfg, weights=sd)
    loss = mae(_to_dev(x), noise=noise.to(DEV))
    loss.backward()
    for k in O.param_keys(sd):
        sd[k].requires_grad_(True)
    inter = {}
    lref = O.vtmae_forward(sd, cfg, x, noise, intermediates=inter)
    lref.backward()
    assert torch.equal(mae.last_masked_indices.cpu(), inter["masked_indices"])
    assert abs(loss.item() - lref.item()) <= 1e-2 * abs(lref.item()), (loss.item(), lref.item())
    named = dict(mae.named_parameters(remove_duplicate=False))
    for k in O.param_keys(sd):
        gr = sd[k].grad
        if gr is None:
            assert named[k].grad is None, k
            continue
        assert _dcos(named[k].grad, gr) >= 0.999, (k, _dcos(named[k].grad, gr))
    with torch.no_grad():
        emb = mae.get_embeddings(_to_dev(x), eval=True)
        eref = O.vtmae_embeddings({k: v.detach() for k, v in sd.items()}, cfg, x)
    assert emb.shape == eref.shape
    assert _dcos(emb, eref) >= 0.9995, _dcos(emb, eref)


@pytest.mark.parametrize("heads,dh,dheads,ddh", _VTMAE_CASES)
def test_vtmae_head_dims_graph_path_matches_eager(heads, dh, dheads, ddh):
    from tests._build import build_product
    B = 4
    cfg, sd, x, noise = _vtmae_case(heads, dh, dheads, ddh, B, seed=3)
    mae_g = build_product(cfg, weights=sd)
    mae_e = build_product(cfg, weights=sd)
    mae_e.use_cuda_graph = False
    for it in range(2):
        for m in (mae_g, mae_e):
            m.zero_grad(set_to_none=True)
        lg = mae_g(_to_dev(x), noise=noise.to(DEV)); lg.backward()
        le = mae_e(_to_dev(x), noise=noise.to(DEV)); le.backward()
        assert torch.equal(lg.detach(), le.detach())
        assert torch.equal(mae_g.last_masked_indices, mae_e.last_masked_indices)
        ge, gg = dict(mae_e.named_parameters()), dict(mae_g.named_parameters())
        for k, p in ge.items():
            assert (p.grad is None) == (gg[k].grad is None), k
            if p.grad is not None:
                assert torch.allclose(gg[k].grad, p.grad, rtol=2e-3, atol=1e-6), k     # fp32 atomics: order only


@pytest.mark.parametrize("heads,dh,dheads,ddh", _VTMAE_CASES)
def test_vtmae_head_dims_fused_train_steps_vs_oracle(heads, dh, dheads, ddh):
    from oracle import vtmae_oracle as O
    from tests._build import build_product
    B = 4
    cfg, sd, x, noise = _vtmae_case(heads, dh, dheads, ddh, B, seed=4)
    mae = build_product(cfg, weights=sd)
    mae.initialize_training({"lr": 1e-4, "batch_size": B})
    st = O.AdamWState()
    xd, nd = _to_dev(x), noise.to(DEV)
    w0 = {k: v.detach().clone() for k, v in sd.items()}
    for it in range(3):
        l = mae.train_step(xd, noise=nd)
        lo, norm, _ = O.train_step(sd, cfg, x, noise, st)
        assert abs(l.item() - lo.item()) <= 1e-2 * abs(lo.item()), (it, l.item(), lo.item())
        assert abs(mae._trainer.state[2].item() - norm.item()) <= 3e-2 * norm.item()
    named = dict(mae.named_parameters())
    for k in ["encoder.transformer.layers.0.0.to_qkv.weight", "decoder.layers.0.0.to_qkv.weight",
              "decoder.layers.1.1.net.1.weight", "to_pixels.weight", "mask_token"]:
        upd_ref = sd[k].detach() - w0[k]
        upd = named[k].detach().cpu() - w0[k]
        assert _dcos(upd, upd_ref) >= 0.99, (k, _dcos(upd, upd_ref))


def test_vtt_dino_dim_head_32_above_256_tokens_vs_oracle():
    """DINO-side VTT with 32-wide heads over three 96 x 96 maps at patch 8 (433 tokens): outputs and every gradient."""
    from oracle import vtt_dino_oracle as VD
    from m3l_b200.vtt import VTT
    cfg = VD.VTTDinoConfig(image_size=(96, 96), tactile_size=(96, 96), image_patch_size=8, tactile_patch_size=8, depth=2,
                           num_register_tokens=1, heads=8, dim_head=32)
    torch.manual_seed(21)
    m = VTT(image_size=cfg.image_size, tactile_size=cfg.tactile_size, image_patch_size=cfg.image_patch_size,
            tactile_patch_size=cfg.tactile_patch_size, dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, mlp_dim=cfg.mlp_dim,
            num_tactiles=cfg.num_tactiles, image_channels=cfg.image_channels, tactile_channels=cfg.tactile_channels,
            dim_head=cfg.dim_head, num_register_tokens=cfg.num_register_tokens, pos_embed_fn="sinusoidal")
    with torch.no_grad():
        m.register_tokens.normal_(0, 0.5)
        for k, p in m.named_parameters():
            if k.endswith(".bias"):
                p.normal_(0, 0.05)
            elif p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.1)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    g = torch.Generator().manual_seed(31)
    B = 2
    x = {"image": torch.rand(B, 12, 96, 96, generator=g), "tactile1": torch.rand(B, 12, 96, 96, generator=g),
         "tactile2": torch.rand(B, 12, 96, 96, generator=g)}
    out = m.forward_features(_to_dev(x), None)
    assert out["x_prenorm"].shape[1] > 256
    for k in sd:
        if sd[k].dtype.is_floating_point and k != "pos_embed.frequency_bands":
            sd[k].requires_grad_(True)
    ref = VD.forward_features(sd, cfg, x, None)
    for k in ("x_norm_regtokens", "x_norm_patchtokens", "x_prenorm"):
        assert out[k].shape == ref[k].shape, k
        assert _dcos(out[k], ref[k]) >= 0.9995, (k, _dcos(out[k], ref[k]))
    w1 = torch.randn(ref["x_norm_patchtokens"].shape, generator=g)
    w2 = torch.randn(ref["x_prenorm"].shape, generator=g)
    ((out["x_norm_patchtokens"] * w1.to(DEV)).sum() + (out["x_norm_regtokens"] ** 2).sum()
     + 0.5 * (out["x_prenorm"] * w2.to(DEV)).sum()).backward()
    ((ref["x_norm_patchtokens"] * w1).sum() + (ref["x_norm_regtokens"] ** 2).sum() + 0.5 * (ref["x_prenorm"] * w2).sum()).backward()
    for k, p in m.named_parameters():
        gr = sd[k].grad
        if gr is None or float(gr.abs().max()) == 0.0:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
        else:
            assert p.grad is not None and _dcos(p.grad, gr) >= 0.999, (k, _dcos(p.grad, gr) if p.grad is not None else None)


def test_standalone_transformer_dim_head_128_under_autograd():
    """m3l_b200.Transformer(dim 256, depth 2, heads 2, dim_head 128) against oracle.vtmae_oracle.transformer."""
    from oracle import vtmae_oracle as O
    from m3l_b200.vtmae import Transformer
    torch.manual_seed(5)
    dim, depth, heads, dh, mlp = 256, 2, 2, 128, 512
    t = Transformer(dim, depth, heads, dh, mlp)
    with torch.no_grad():
        for k, p in t.named_parameters():
            if k.endswith(".bias"):
                p.normal_(0, 0.05)
            elif p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.1)
    sd = {"t." + k: v.detach().clone().requires_grad_(True) for k, v in t.state_dict().items()}
    t = t.to(DEV)
    B, n = 3, 150
    x = torch.randn(B, n, dim)
    xd = x.to(DEV).requires_grad_(True)
    y = t(xd)
    xr = x.clone().requires_grad_(True)
    yr = O.transformer(xr, sd, "t", depth, heads, dh)
    assert y.shape == yr.shape
    assert _dcos(y, yr) >= 0.9995, _dcos(y, yr)
    w = torch.randn(yr.shape)
    (y.float() * w.to(DEV)).sum().backward()
    (yr * w).sum().backward()
    assert _dcos(xd.grad, xr.grad) >= 0.999, _dcos(xd.grad, xr.grad)
    for k, p in t.named_parameters():
        assert _dcos(p.grad, sd["t." + k].grad) >= 0.999, (k, _dcos(p.grad, sd["t." + k].grad))
