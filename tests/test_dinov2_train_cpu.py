"""Fine-tuning DinoV2 (CPU part): the oracle's gradients against the `transformers` implementation of the same network,
the LayerScale fold / unfold algebra the kernel path uses, and the position-table backward."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import dinov2_oracle as DO


def _hf_grads_as_hub(m):
    g = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in m.named_parameters()}
    return DO.hf_to_hub_state_dict(g)


@pytest.mark.parametrize("grid,table_grid", [(5, 5), (5, 37), (16, 16), (16, 37)])
def test_oracle_gradients_match_transformers(grid, table_grid):
    """grid == table_grid: no position interpolation; table_grid 37 (the 518 x 518 pre-training table): bicubic."""
    tr = pytest.importorskip("transformers")
    torch.manual_seed(0)
    cfg = tr.Dinov2WithRegistersConfig(hidden_size=384, num_hidden_layers=2, num_attention_heads=6, mlp_ratio=4,
                                       patch_size=14, image_size=14 * table_grid, num_register_tokens=4,
                                       layerscale_value=1.0)
    m = tr.Dinov2WithRegistersModel(cfg).eval()
    sd = DO.random_state_dict(depth=2, grid=table_grid, seed=3, ls_init=0.3)
    hub = DO.hf_to_hub_state_dict(m.state_dict())
    sd["mask_token"] = hub["mask_token"]
    assert set(sd) == set(hub)
    with torch.no_grad():                       # load the random hub weights into the transformers model
        hf = m.state_dict()
        D = 384
        hf["embeddings.cls_token"].copy_(sd["cls_token"]); hf["embeddings.position_embeddings"].copy_(sd["pos_embed"])
        hf["embeddings.register_tokens"].copy_(sd["register_tokens"])
        hf["embeddings.patch_embeddings.projection.weight"].copy_(sd["patch_embed.proj.weight"])
        hf["embeddings.patch_embeddings.projection.bias"].copy_(sd["patch_embed.proj.bias"])
        hf["layernorm.weight"].copy_(sd["norm.weight"]); hf["layernorm.bias"].copy_(sd["norm.bias"])
        for i in range(2):
            p, q = f"encoder.layer.{i}.", f"blocks.{i}."
            a = p + "attention.attention."
            for j, nm in enumerate(("query", "key", "value")):
                hf[a + nm + ".weight"].copy_(sd[q + "attn.qkv.weight"][j * D:(j + 1) * D])
                hf[a + nm + ".bias"].copy_(sd[q + "attn.qkv.bias"][j * D:(j + 1) * D])
            hf[p + "attention.output.dense.weight"].copy_(sd[q + "attn.proj.weight"])
            hf[p + "attention.output.dense.bias"].copy_(sd[q + "attn.proj.bias"])
            hf[p + "layer_scale1.lambda1"].copy_(sd[q + "ls1.gamma"]); hf[p + "layer_scale2.lambda1"].copy_(sd[q + "ls2.gamma"])
            for nm in ("norm1", "norm2", "mlp.fc1", "mlp.fc2"):
                hf[p + nm + ".weight"].copy_(sd[q + nm + ".weight"]); hf[p + nm + ".bias"].copy_(sd[q + nm + ".bias"])
    gen = torch.Generator().manual_seed(1)
    x = torch.rand(2, 3, 14 * grid, 14 * grid, generator=gen)
    cot = torch.randn(2, 1 + 4 + grid * grid, D, generator=gen)
    out = m(pixel_values=x)
    ((out.last_hidden_state * cot).sum() + out.pooler_output.square().sum()).backward()
    want = _hf_grads_as_hub(m)
    leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    tok = DO.dinov2_forward(leaves, x, return_tokens=True)
    ((tok * cot).sum() + tok[:, 0].square().sum()).backward()
    for k, v in leaves.items():
        if k == "mask_token":
            assert v.grad is None
            continue
        err = (v.grad - want[k]).abs().max() / want[k].abs().max().clamp_min(1e-12)
        assert err <= 1e-5, (k, float(err))


def test_layerscale_fold_unfold_algebra():
    """y = x (g o W)^T + g o b: dW = g o dW', db = g o db', dg = rowsum(W o dW') + b o db' (what csrc/layerscale.cu
    computes), with a non-unit, non-constant g."""
    gen = torch.Generator().manual_seed(0)
    rows, cols, M = 48, 80, 33
    W = torch.randn(rows, cols, generator=gen, dtype=torch.float64).requires_grad_(True)
    b = torch.randn(rows, generator=gen, dtype=torch.float64).requires_grad_(True)
    g = (0.5 + torch.rand(rows, generator=gen, dtype=torch.float64)).mul(0.1).requires_grad_(True)
    x = torch.randn(M, cols, generator=gen, dtype=torch.float64)
    cot = torch.randn(M, rows, generator=gen, dtype=torch.float64)
    Wf, bf = g[:, None] * W, g * b
    Wf.retain_grad(); bf.retain_grad()
    ((x @ Wf.T + bf) * cot).sum().backward()
    dWf, dbf = Wf.grad, bf.grad
    torch.testing.assert_close(W.grad, g.detach()[:, None] * dWf, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(b.grad, g.detach() * dbf, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(g.grad, (W.detach() * dWf).sum(1) + b.detach() * dbf, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("table_grid,gh,gw", [(37, 16, 16), (37, 5, 5), (5, 5, 5), (4, 3, 5)])
def test_pos_table_backward_matches_autograd(table_grid, gh, gw):
    from m3l_b200.dinov2 import DinoV2, pos_table_bwd
    m = DinoV2(img_size=14 * table_grid, depth=1)
    gen = torch.Generator().manual_seed(2)
    with torch.no_grad():
        m.pos_embed.copy_(torch.randn(m.pos_embed.shape, generator=gen))
    pe = m.pos_embed.detach().clone().requires_grad_(True)   # _pos_table detaches: its graph is rebuilt on a leaf
    n_pos = pe.shape[1] - 1
    if n_pos == gh * gw and gh == gw:
        rows = pe[0, 1:]
    else:
        g = int(math.sqrt(n_pos))
        p = pe[:, 1:].reshape(1, g, g, 384).permute(0, 3, 1, 2)
        p = F.interpolate(p, size=(gh, gw), mode="bicubic", align_corners=False, antialias=True)
        rows = p.permute(0, 2, 3, 1).reshape(gh * gw, 384)
    assert torch.equal(rows.detach(), m._pos_table(gh, gw)[1:])
    cot = torch.randn(gh * gw, 384, generator=gen)
    (rows * cot).sum().backward()
    torch.testing.assert_close(pos_table_bwd(cot, n_pos, gh, gw), pe.grad[0, 1:], rtol=1e-5, atol=1e-6)


def test_fine_tuning_needs_cuda_parameters():
    """A training-mode module with trainable CPU parameters raises instead of falling back to eager torch."""
    from m3l_b200.dinov2 import DinoV2
    from m3l_b200._lib import M3LError
    m = DinoV2(img_size=70, depth=1).train()
    with pytest.raises(M3LError, match="fine-tuning needs contiguous fp32 CUDA parameters"):
        m(torch.rand(1, 3, 70, 70))
