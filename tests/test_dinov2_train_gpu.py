"""Fine-tuning DinoV2 on the sm_100a kernels, against autograd through the CPU oracle (oracle/dinov2_oracle.py).

Gradients are compared per parameter by cosine; forward outputs with the tolerances of tests/test_dinov2.py.
Gradients are summed with fp32 atomics in the wgrad / column-sum / LayerNorm kernels, so two runs of the same
backward agree to rounding, not bit for bit; forward outputs are bit-identical."""
import pytest
import torch

from oracle import dinov2_oracle as DO

DEV = "cuda"
pytestmark = pytest.mark.gpu


def _cos(a, b):
    a, b = a.detach().double().flatten(), b.detach().double().flatten()
    return float(a @ b / (a.norm() * b.norm() + 1e-300))


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def _model(table_grid=5, depth=4, seed=1):
    from m3l_b200.dinov2 import DinoV2
    sd = DO.random_state_dict(grid=table_grid, depth=depth, seed=seed, ls_init=0.3)
    sd["mask_token"] = torch.zeros(1, 384)
    m = DinoV2(img_size=14 * table_grid, depth=depth)
    m.load_state_dict(sd)
    return m.to(DEV).train(), sd


def _inputs(B, grid, return_tokens, seed=3):
    gen = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, 14 * grid, 14 * grid, generator=gen)
    cot = torch.randn((B, 5 + grid * grid, 384) if return_tokens else (B, 384), generator=gen)
    return x, cot


def _oracle(sd, x, cot, return_tokens=False):
    leaves = {k: v.clone().requires_grad_(k != "mask_token") for k, v in sd.items()}
    out = DO.dinov2_forward(leaves, x, return_tokens=return_tokens)
    (out * cot).sum().backward()
    return out.detach(), {k: v.grad for k, v in leaves.items() if k != "mask_token"}


def _grads(m):
    return {k: (None if p.grad is None else p.grad.detach().cpu().clone()) for k, p in m.named_parameters()}


def _launches(eager_depth):
    """Kernels of the frozen forward: patchify, patch GEMM, token assembly, 7 per block, final LayerNorm."""
    return 3 + 7 * eager_depth + 1


@pytest.mark.parametrize("table_grid,grid,depth,B,return_tokens", [
    (5, 5, 12, 4, False),          # n = 30: the n <= 256 attention kernels
    (16, 16, 12, 2, False),        # n = 261: the long attention kernels
    (37, 16, 4, 2, False),         # 518-table model fed 224 x 224: position interpolation backward
    (5, 5, 4, 3, True),            # all tokens, random cotangent
])
def test_gradients_vs_oracle(table_grid, grid, depth, B, return_tokens):
    m, sd = _model(table_grid, depth)
    x, cot = _inputs(B, grid, return_tokens)
    ref, want = _oracle(sd, x, cot, return_tokens)
    out = m(x.to(DEV), return_tokens=return_tokens)
    assert out.grad_fn is not None
    assert _cos(out.cpu(), ref) >= 0.999
    assert (out.detach().cpu() - ref).abs().max() <= 0.06 * ref.abs().max()
    (out * cot.to(DEV)).sum().backward()
    got = _grads(m)
    assert got["mask_token"] is None
    worst = min((_cos(got[k], want[k]), k) for k in want)
    print("min gradient cosine", worst)
    assert worst[0] >= 0.999, worst


def test_partial_fine_tuning_last_two_blocks():
    from m3l_b200 import ops
    m, sd = _model(5, 4)
    m.use_cuda_graph = False
    x, cot = _inputs(4, 5, False)
    x, cot = x.to(DEV), cot.to(DEV)
    out = m(x)
    with ops.LaunchCounter() as full:
        (out * cot).sum().backward()
    g_full = _grads(m)
    m.zero_grad(set_to_none=True)
    for k, p in m.named_parameters():
        p.requires_grad_(k.startswith(("blocks.2.", "blocks.3.")))
    out = m(x)
    with ops.LaunchCounter() as part:
        (out * cot).sum().backward()
    g = _grads(m)
    for k, p in m.named_parameters():
        if p.requires_grad:
            assert g[k] is not None and _rel(g[k], g_full[k]) <= 1e-3, k
        else:
            assert g[k] is None, k
    assert part.count < full.count, (part.count, full.count)


def test_frozen_path_is_unchanged():
    from m3l_b200 import ops
    m, _ = _model(5, 4)
    x, _ = _inputs(3, 5, False)
    x = x.to(DEV)
    m.eval()
    ref = m(x)
    assert ref.grad_fn is None
    m.use_cuda_graph = False
    with ops.LaunchCounter() as lc:
        assert m(x).grad_fn is None
    assert lc.count == _launches(4)
    m.use_cuda_graph = True
    with ops.LaunchCounter() as lc:
        assert torch.equal(m(x), ref)
    assert lc.count == 0                                   # replayed from the captured frozen graph
    m.train()
    with torch.no_grad(), ops.LaunchCounter() as lc:
        assert torch.equal(m(x), ref)
    assert lc.count == 0
    for p in m.parameters():
        p.requires_grad_(False)
    with ops.LaunchCounter() as lc:
        out = m(x)
    assert out.grad_fn is None and torch.equal(out, ref) and lc.count == 0
    for p in m.parameters():
        p.requires_grad_(True)
    for graph in (True, False):                            # the fine-tuning forward computes the same bits
        m.use_cuda_graph = graph
        out = m(x)
        assert out.grad_fn is not None and torch.equal(out.detach(), ref)
        tok = m(x, return_tokens=True)
        with torch.no_grad():
            assert torch.equal(tok.detach(), m(x, return_tokens=True))


def test_graph_replay_matches_eager():
    m, _ = _model(5, 4)
    x, cot = _inputs(4, 5, False)
    x, cot = x.to(DEV), cot.to(DEV)
    m.use_cuda_graph = False
    out_e = m(x)
    (out_e * cot).sum().backward()
    g_e = _grads(m)
    m.zero_grad(set_to_none=True)
    m.use_cuda_graph = True
    for _ in range(2):                                     # capture, then replay
        m.zero_grad(set_to_none=True)
        out_g = m(x)
        (out_g * cot).sum().backward()
        assert torch.equal(out_g.detach(), out_e.detach())
        g_g = _grads(m)
        for k in g_e:
            if g_e[k] is not None:
                assert _rel(g_g[k], g_e[k]) <= 1e-3, k


def test_graph_survives_in_place_weight_updates():
    """Three AdamW steps (torch optimizer, lr 1e-4) replayed without re-capture, tracked against the oracle; then a
    large in-place edit of the weights is picked up by the next replay."""
    m, sd = _model(5, 4)
    x, cot = _inputs(4, 5, False)
    xd, cd = x.to(DEV), cot.to(DEV)
    leaves = {k: v.clone().requires_grad_(k != "mask_token") for k, v in sd.items()}
    opt = torch.optim.AdamW([p for p in m.parameters() if p.requires_grad and p is not m.mask_token], lr=1e-4)
    opt_ref = torch.optim.AdamW([v for k, v in leaves.items() if k != "mask_token"], lr=1e-4)
    p0 = {k: v.detach().clone() for k, v in sd.items()}
    ents = None
    for step in range(3):
        out = m(xd)
        (out * cd).sum().backward()
        opt.step(); opt.zero_grad(set_to_none=True)
        ref = DO.dinov2_forward(leaves, x)
        (ref * cot).sum().backward()
        opt_ref.step(); opt_ref.zero_grad(set_to_none=True)
        assert _cos(out.detach().cpu(), ref.detach()) >= 0.999
        cur = list(m.__dict__["_train_ops"]["graphs"].values())
        assert ents is None or (len(cur) == 1 and cur[0] is ents[0])
        ents = cur
    params = dict(m.named_parameters())
    dg = torch.cat([(params[k].detach().cpu() - p0[k]).flatten() for k in p0 if k != "mask_token"])
    dr = torch.cat([(leaves[k].detach() - p0[k]).flatten() for k in p0 if k != "mask_token"])
    print("AdamW update cosine", _cos(dg, dr))
    assert _cos(dg, dr) >= 0.99                            # 0.9986 measured on a B200
    with torch.no_grad():
        m.blocks[-1].mlp.fc2.weight.mul_(1.5)
        m.blocks[0].ls1.gamma.add_(0.25)
        m.pos_embed.mul_(0.5)
    out = m(xd)
    assert m.__dict__["_train_ops"]["graphs"] and list(m.__dict__["_train_ops"]["graphs"].values())[0] is ents[0]
    m.eval()
    with torch.no_grad():
        assert torch.equal(out.detach(), m(xd))


def test_superseded_backward_raises_and_two_backwards_accumulate():
    from m3l_b200._lib import M3LError
    m, _ = _model(5, 2)
    x, cot = _inputs(2, 5, False)
    x, cot = x.to(DEV), cot.to(DEV)
    out1 = m(x)
    out2 = m(x)
    with pytest.raises(M3LError, match="overwritten by a newer forward"):
        (out1 * cot).sum().backward()
    m.zero_grad(set_to_none=True)
    (out2 * cot).sum().backward()
    g1 = _grads(m)
    (m(x) * cot).sum().backward()
    g2 = _grads(m)
    for k in g1:
        if g1[k] is not None:
            assert _rel(g2[k], 2 * g1[k]) <= 1e-3, k


def test_layerscale_kernels():
    from m3l_b200 import ops
    gen = torch.Generator().manual_seed(5)
    rows, cols = 384, 1536
    w = torch.randn(rows, cols, generator=gen).to(DEV)
    b = torch.randn(rows, generator=gen).to(DEV)
    g = (0.5 + torch.rand(rows, generator=gen)).mul(0.1).to(DEV)
    wf = torch.empty(rows, cols, dtype=torch.bfloat16, device=DEV)
    wf_t = torch.empty(cols, rows, dtype=torch.bfloat16, device=DEV)
    bf = torch.empty(rows, device=DEV)
    ops.layerscale_fold(w, b, g, wf, wf_t, bf)
    want = (g[:, None] * w).to(torch.bfloat16)
    assert torch.equal(wf, want) and torch.equal(wf_t, want.t().contiguous()) and torch.equal(bf, g * b)
    ops.layerscale_fold(w, None, None, wf, wf_t)
    assert torch.equal(wf, w.to(torch.bfloat16)) and torch.equal(wf_t, w.t().to(torch.bfloat16))
    dwf = torch.randn(rows, cols, generator=gen).to(DEV)
    dbf = torch.randn(rows, generator=gen).to(DEV)
    dw, db, dg = torch.empty_like(w), torch.empty_like(b), torch.empty_like(g)
    ops.layerscale_unfold(dwf, dbf, w, b, g, dw, db, dg)
    torch.testing.assert_close(dw, g[:, None] * dwf, rtol=1e-6, atol=0)
    torch.testing.assert_close(db, g * dbf, rtol=1e-6, atol=0)
    want_g = (w.double() * dwf.double()).sum(1) + b.double() * dbf.double()
    torch.testing.assert_close(dg.double(), want_g, rtol=1e-4, atol=1e-3)


def test_extractor_keeps_dino_frozen_in_training_mode():
    from m3l_b200.dinov2 import DinoV2, DinoCatMAEExtractor
    from oracle import vtmae_oracle as O
    from tests._build import build_product
    F, dim = 4, 384
    cfg = O.VTMAEConfig(image_size=(70, 70), tactile_size=(70, 70), image_patch_size=14, tactile_patch_size=14, dim=dim,
                        depth=2, heads=4, mlp_dim=2 * dim, decoder_dim=dim, decoder_depth=1, decoder_heads=4,
                        masking_ratio=0.8)
    mae = build_product(cfg, weights=O.init_state_dict(cfg, seed=5))
    dsd = DO.random_state_dict(grid=5, depth=3, seed=2)
    dsd["mask_token"] = torch.zeros(1, 384)
    dino = DinoV2(img_size=70, depth=3)
    dino.load_state_dict(dsd)
    dino = dino.to(DEV)
    ext = DinoCatMAEExtractor(None, dino, mae, dim, False, F).to(DEV).train()
    assert dino.training and all(p.requires_grad for p in dino.parameters())
    gen = torch.Generator().manual_seed(4)
    B = 3
    obs = {"image": torch.rand(B, F, 70, 70, 3, generator=gen), "tactile": torch.rand(B, F, 6, 70, 70, generator=gen) * 2 - 1}
    out = ext(obs)
    out.square().sum().backward()
    assert all(p.grad is None for p in dino.parameters())
    assert ext.mlp[0].weight.grad is not None
