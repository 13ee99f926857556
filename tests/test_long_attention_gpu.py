"""GPU: the attention kernels for sequences of any length (csrc/attention_long.cu) against a plain fp32 torch statement,
against the n <= 256 kernels where both apply, and through the models whose sequences exceed 256 tokens."""
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"


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


def _attn_ref(qkv, B, n, H, scale):
    q, k, v = qkv.float().reshape(B, n, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-1, -2)) * scale
    return (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B * n, H * 64), torch.logsumexp(s, -1)


def _check_vs_ref(ops, qkv, B, n, H, seed=11):
    scale = 64 ** -0.5
    out, lse = ops.attention_long_fwd(qkv, B, n, H, 64, scale)
    qr = qkv.float().requires_grad_(True)
    oref, lref = _attn_ref(qr, B, n, H, scale)
    assert torch.isfinite(out.float()).all() and torch.isfinite(lse).all()
    assert rel_err(out, oref) < 2e-2
    assert (lse - lref).abs().max().item() < 2e-2
    g = torch.Generator(device=DEV).manual_seed(seed)
    dout = torch.randn(B * n, H * 64, device=DEV, generator=g).bfloat16()
    oref.backward(dout.float())
    inner = H * 64
    delta = (dout.float() * out.float()).reshape(B * n, H, 64).sum(-1).contiguous()
    for d in (None, delta):
        dqkv = ops.attention_long_bwd(qkv, out, dout, lse, B, n, H, 64, scale, delta=d)
        assert torch.isfinite(dqkv.float()).all()
        for name, sl in (("dq", slice(0, inner)), ("dk", slice(inner, 2 * inner)), ("dv", slice(2 * inner, 3 * inner))):
            assert cos(dqkv[:, sl], qr.grad[:, sl]) > 0.999, (name, d is None)
            assert rel_err(dqkv[:, sl], qr.grad[:, sl]) < 5e-2, (name, d is None)
    return out, lse


@pytest.mark.parametrize("B,n,H", [(2, 257, 1), (3, 261, 6), (2, 300, 4), (2, 383, 2), (1, 384, 4), (2, 385, 3),
                                   (1, 1000, 2), (2, 1374, 6), (1, 4096, 1),
                                   (64, 261, 6)])          # more (sample, head, tile) items than SMs
def test_long_attention_vs_fp32(ops, B, n, H):
    torch.manual_seed(7)
    qkv = torch.randn(B * n, 3 * H * 64, device=DEV).bfloat16()
    _check_vs_ref(ops, qkv, B, n, H)


@pytest.mark.parametrize("B,n,H,late", [(2, 300, 2, True), (1, 1000, 3, True), (2, 385, 2, False)])
def test_online_softmax_rescaling(ops, B, n, H, late):
    """late=True: the largest score of many rows sits in the LAST key tile (spike keys scaled up), so the running max
    grows late and O must be rescaled; late=False: large-magnitude scores everywhere (qkv x 4)."""
    torch.manual_seed(3)
    x = torch.randn(B, n, 3, H, 64, device=DEV)
    if late:
        last0 = (n - 1) // 128 * 128
        spikes = torch.arange(last0, n, 7, device=DEV)
        # every query leans along u, the spike keys (tail tile only) are 40 u: scaled scores ~10 there against ~3 for
        # the largest ordinary ones, a jump of more than the kernel's rescaling threshold (8 in log2 units)
        u = torch.nn.functional.normalize(torch.randn(H, 64, device=DEV), dim=-1)
        x[:, :, 0] += 2.0 * u
        x[:, spikes, 1] = 40.0 * u
    else:
        x = x * 4.0
    qkv = x.reshape(B * n, 3 * H * 64).bfloat16().contiguous()
    _check_vs_ref(ops, qkv, B, n, H)


@pytest.mark.parametrize("n", [17, 130, 192, 256])
def test_long_kernels_agree_with_short_kernels(ops, n):
    torch.manual_seed(5)
    B, H, scale = 3, 4, 64 ** -0.5
    qkv = torch.randn(B * n, 3 * H * 64, device=DEV).bfloat16()
    o1, l1 = ops.attention_fwd(qkv, B, n, H, 64, scale)
    o2, l2 = ops.attention_long_fwd(qkv, B, n, H, 64, scale)
    assert rel_err(o2, o1) < 1e-2 and (l2 - l1).abs().max().item() < 1e-2
    dout = torch.randn(B * n, H * 64, device=DEV).bfloat16()
    d1 = ops.attention_bwd(qkv, o1, dout, l1, B, n, H, 64, scale)
    d2 = ops.attention_long_bwd(qkv, o1, dout, l1, B, n, H, 64, scale)
    assert cos(d2, d1) > 0.9999 and rel_err(d2, d1) < 2e-2


def test_mha_selects_by_length(ops):
    """n <= 256 runs the short kernels bit for bit; above, the long ones."""
    torch.manual_seed(6)
    scale = 64 ** -0.5
    for n, short in ((256, True), (257, False)):
        B, H = 2, 2
        qkv = torch.randn(B * n, 3 * H * 64, device=DEV).bfloat16()
        o, l = ops.mha_fwd(qkv, B, n, H, 64, scale)
        ref_f = ops.attention_fwd if short else ops.attention_long_fwd
        ref_b = ops.attention_bwd if short else ops.attention_long_bwd
        o_r, l_r = ref_f(qkv, B, n, H, 64, scale)
        assert torch.equal(o, o_r) and torch.equal(l, l_r)
        dout = torch.randn_like(o)
        assert torch.equal(ops.mha_bwd(qkv, o, dout, l, B, n, H, 64, scale), ref_b(qkv, o, dout, l, B, n, H, 64, scale))


@pytest.mark.parametrize("B,n,H", [(2, 1374, 6), (64, 261, 6)])
def test_long_attention_is_deterministic(ops, B, n, H):
    torch.manual_seed(9)
    scale = 64 ** -0.5
    qkv = torch.randn(B * n, 3 * H * 64, device=DEV).bfloat16()
    dout = torch.randn(B * n, H * 64, device=DEV).bfloat16()
    runs = []
    for _ in range(2):
        o, l = ops.attention_long_fwd(qkv, B, n, H, 64, scale)
        runs.append((o, l, ops.attention_long_bwd(qkv, o, dout, l, B, n, H, 64, scale)))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("n", [261, 1374])
def test_no_writes_past_the_end(ops, n):
    """Outputs are prefixes of larger sentinel-filled buffers: rows beyond B*n (and heads beyond H in lse) stay intact."""
    torch.manual_seed(4)
    B, H, scale, extra = 2, 3, 64 ** -0.5, 200
    inner = H * 64
    qkv = torch.randn(B * n, 3 * inner, device=DEV).bfloat16()
    sentinel = -1234.0
    out_buf = torch.full(((B * n + extra) * inner,), sentinel, device=DEV).bfloat16()
    lse_buf = torch.full((B * H * n + extra,), sentinel, device=DEV)
    out = out_buf[:B * n * inner].view(B * n, inner)
    lse = lse_buf[:B * H * n].view(B, H, n)
    ops.attention_long_fwd(qkv, B, n, H, 64, scale, out=out, lse=lse)
    assert (out_buf[B * n * inner:] == sentinel).all() and (lse_buf[B * H * n:] == sentinel).all()
    o_ref, l_ref = _attn_ref(qkv, B, n, H, scale)
    assert rel_err(out, o_ref) < 2e-2 and (lse - l_ref).abs().max().item() < 2e-2
    dq_buf = torch.full(((B * n + extra) * 3 * inner,), sentinel, device=DEV).bfloat16()
    dqkv = dq_buf[:B * n * 3 * inner].view(B * n, 3 * inner)
    dout = torch.randn(B * n, inner, device=DEV).bfloat16()
    ops.attention_long_bwd(qkv, out, dout, lse, B, n, H, 64, scale, dqkv=dqkv)
    assert (dq_buf[B * n * 3 * inner:] == sentinel).all()
    assert torch.isfinite(dqkv.float()).all()


def test_errors_are_loud(ops):
    from m3l_b200._lib import M3LError
    qkv = torch.randn(2 * 300, 3 * 2 * 32, device=DEV).bfloat16()
    with pytest.raises(M3LError, match="status 3"):
        ops.attention_long_fwd(qkv, 2, 300, 2, 32, 0.125)


def test_opcheck_long_attention():
    import m3l_b200.torch_ops  # noqa: F401  (registers torch.ops.m3l)
    OPS = torch.ops.m3l
    torch.manual_seed(2)
    B, n, H = 2, 300, 2
    qkv = torch.randn(B * n, 3 * H * 64, device=DEV).bfloat16()
    torch.library.opcheck(OPS.attention_long_fwd.default, (qkv, B, n, H, 64, 0.125))
    o, lse = OPS.attention_long_fwd(qkv, B, n, H, 64, 0.125)
    torch.library.opcheck(OPS.attention_long_bwd.default, (qkv, o, torch.randn_like(o), lse, B, n, H, 64, 0.125))


# ------------------------------------------------------------------------------ models above 256 tokens
def _dcos(a, b):
    a, b = a.detach().double().flatten().cpu(), b.detach().double().flatten().cpu()
    return float(a @ b / (a.norm() * b.norm() + 1e-300))


@pytest.mark.parametrize("size", [224, 518])
def test_dinov2_at_its_own_resolutions_vs_oracle(size):
    """The default DinoV2 (518 x 518, 37 x 37 position table): 224 x 224 input (n = 261, table interpolated to 16 x 16)
    and 518 x 518 (n = 1374, no interpolation); the graph-replayed call is bit-identical to the eager one."""
    from oracle import dinov2_oracle as DO
    from m3l_b200.dinov2 import DinoV2
    sd = DO.random_state_dict(grid=37, seed=1)
    sd["mask_token"] = torch.zeros(1, 384)
    m = DinoV2()
    m.load_state_dict(sd)
    m = m.to(DEV).eval()
    gen = torch.Generator().manual_seed(3)
    B = 2
    x = torch.rand(B, 3, size, size, generator=gen)
    ref = DO.dinov2_forward(sd, x)
    got = m(x.to(DEV))
    assert got.shape == (B, 384) and got.dtype == torch.float32
    assert _dcos(got, ref) >= 0.999, _dcos(got, ref)
    assert (got.cpu() - ref).abs().max() <= 0.06 * ref.abs().max()
    m.use_cuda_graph = False
    assert torch.equal(m(x.to(DEV)), got)


def _vtmae_384_case(B, seed):
    from oracle import vtmae_oracle as O
    cfg = O.VTMAEConfig(image_size=(128, 128), image_patch_size=8, depth=2, decoder_depth=2)
    assert cfg.n_img + 2 * cfg.n_tac == 384
    sd = O.init_state_dict(cfg, seed=seed)
    gen = torch.Generator().manual_seed(seed + 50)
    x = {"image": torch.rand(B, 12, 128, 128, generator=gen), "tactile1": torch.rand(B, 12, 32, 32, generator=gen),
         "tactile2": torch.rand(B, 12, 32, 32, generator=gen)}
    noise = O.tie_free_noise(B, 384, gen, [cfg.n_img, cfg.n_tac, cfg.n_tac])
    return cfg, sd, x, noise


def _to_dev(x):
    return {k: v.to(DEV) for k, v in x.items()}


def test_vtmae_384_tokens_vs_oracle():
    """128 x 128 image at patch 8 + two 32 x 32 tactile maps at patch 4: the decoder (and get_embeddings' encoder) see
    384 tokens.  Mask indices bit-exact, loss, every gradient, embeddings."""
    from oracle import vtmae_oracle as O
    from tests._build import build_product
    B = 4
    cfg, sd, x, noise = _vtmae_384_case(B, seed=1)
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
    assert emb.shape == eref.shape == (B, 384, cfg.dim)
    assert _dcos(emb, eref) >= 0.9995, _dcos(emb, eref)


def test_vtmae_384_tokens_graph_path_matches_eager():
    from tests._build import build_product
    B = 4
    cfg, sd, x, noise = _vtmae_384_case(B, seed=3)
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


def test_vtmae_384_tokens_fused_train_steps_vs_oracle():
    from oracle import vtmae_oracle as O
    from tests._build import build_product
    B = 4
    cfg, sd, x, noise = _vtmae_384_case(B, seed=4)
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
    for k in ["decoder.layers.0.0.to_qkv.weight", "decoder.layers.1.1.net.1.weight", "to_pixels.weight", "mask_token"]:
        upd_ref = sd[k].detach() - w0[k]
        upd = named[k].detach().cpu() - w0[k]
        assert _dcos(upd, upd_ref) >= 0.99, (k, _dcos(upd, upd_ref))


@pytest.mark.parametrize("regs,n_masks,keep", [(1, 0, 0), (2, 1, 120)])
def test_vtt_dino_above_256_tokens_vs_oracle(regs, n_masks, keep):
    """DINO-side VTT over three 96 x 96 maps at patch 8 (3 x 144 patch tokens): outputs and every gradient."""
    from oracle import vtt_dino_oracle as VD
    from m3l_b200.vtt import VTT
    cfg = VD.VTTDinoConfig(image_size=(96, 96), tactile_size=(96, 96), image_patch_size=8, tactile_patch_size=8, depth=2,
                           num_register_tokens=regs, heads=4)
    torch.manual_seed(20 + regs)
    m = VTT(image_size=cfg.image_size, tactile_size=cfg.tactile_size, image_patch_size=cfg.image_patch_size,
            tactile_patch_size=cfg.tactile_patch_size, dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, mlp_dim=cfg.mlp_dim,
            num_tactiles=cfg.num_tactiles, image_channels=cfg.image_channels, tactile_channels=cfg.tactile_channels,
            dim_head=cfg.dim_head, num_register_tokens=cfg.num_register_tokens, pos_embed_fn="sinusoidal")
    with torch.no_grad():
        if m.register_tokens is not None:
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
    masks = [torch.stack([torch.randperm(cfg.n_img, generator=g)[:keep] for _ in range(B)]) for _ in range(n_masks)] or None
    out = m.forward_features(_to_dev(x), [mk.to(DEV) for mk in masks] if masks else None)
    assert out["x_prenorm"].shape[1] > 256
    for k in sd:
        if sd[k].dtype.is_floating_point and k != "pos_embed.frequency_bands":
            sd[k].requires_grad_(True)
    ref = VD.forward_features(sd, cfg, x, masks)
    for k in ("x_norm_regtokens", "x_norm_patchtokens", "x_prenorm"):
        assert out[k].shape == ref[k].shape, k
        if out[k].numel():
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
