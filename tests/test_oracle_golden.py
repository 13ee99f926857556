"""CPU: the oracle restatement reproduces the golden vectors frozen from the unmodified reference."""
import pytest
import torch

from oracle import vtmae_oracle as O
from tests._golden import CASES, VTT_DINO_CASES, Golden, VttDinoGolden


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name):
    g = Golden(name)
    cfg, sd, x, noise = g.cfg, g.weights(), g.inputs(), g.noise()
    st = O.AdamWState()
    inter = {}
    keys = O.param_keys(sd)
    for k in keys:
        sd[k].requires_grad_(True)
    loss = O.vtmae_forward(sd, cfg, x, noise, intermediates=inter)
    # integer results: bit-exact
    assert torch.equal(inter["masked_indices"], g.t("masked_indices"))
    assert torch.equal(inter["unmasked_indices"], g.t("unmasked_indices"))
    # fp32 CPU vs fp32 CPU of the same op sequence: tight tolerance (summation order of in-place adds)
    assert torch.allclose(loss.detach(), g.t("loss"), rtol=1e-6, atol=0)
    for k in ("enc_in", "encoded", "decoded"):
        assert torch.allclose(inter[k].detach(), g.t(k), rtol=1e-5, atol=1e-5), k
    loss.backward()
    present = g.grad_present()
    for k, gn in g.grad_norms().items():
        if not present[k]:
            assert sd[k].grad is None or float(sd[k].grad.abs().max()) == 0.0, k
        else:
            assert abs(float(sd[k].grad.double().norm()) - gn) <= 1e-4 * max(gn, 1e-6), k
    for k, gr in g.full_grads().items():
        assert torch.allclose(sd[k].grad, gr, rtol=1e-4, atol=1e-7), k
    # one clip + AdamW step
    grads = {k: (sd[k].grad if present.get(k, True) else None) for k in keys}
    total = O.clip_and_adamw(sd, grads, st)
    assert torch.allclose(total, g.t("grad_total_norm"), rtol=1e-5)
    # A first AdamW step moves a weight by lr * g / (|g| + eps), g the clipped gradient.  Entries with |g| far below
    # eps = 1e-8 are rounding noise of a cancelling sum (~1e-10, their value set by the CPU's summation order: thread
    # count, SIMD width), which that step amplifies by lr / eps.  So the bound adds a gradient error of 1e-9 carried
    # through the step, lr * eps * 1e-9 / (|g| + eps)^2: ~1e-9 wherever |g| >> eps, lr / 10 where |g| << eps.
    coef = min(1.0, 0.5 / (float(total) + 1e-6))
    for k, w in g.after().items():
        gr = grads[k]
        carried = 0.0 if gr is None else 1e-4 * 1e-8 * 1e-9 / (gr.abs() * coef + 1e-8) ** 2
        assert ((sd[k].detach() - w).abs() <= 1e-7 + 1e-6 * w.abs() + carried).all(), k
    with torch.no_grad():
        loss2 = O.vtmae_forward(sd, cfg, x, noise)
    assert torch.allclose(loss2, g.t("loss_after_step"), rtol=1e-5)


@pytest.mark.parametrize("name", CASES)
def test_oracle_embeddings_golden(name):
    g = Golden(name)
    with torch.no_grad():
        emb = O.vtmae_embeddings(g.weights(), g.cfg, g.inputs())
        assert torch.allclose(emb[:1], g.t("embeddings"), rtol=1e-5, atol=1e-5)
        if g.has("embeddings_vision_only"):
            emb = O.vtmae_embeddings(g.weights(), g.cfg, g.inputs(), use_tactile=False)
            assert torch.allclose(emb[:1], g.t("embeddings_vision_only"), rtol=1e-5, atol=1e-5)


def test_mask_counts_python_float_truncation():
    # pretrain_models.py:223-227 on the canonical and the DINO-tac geometry (SURVEY.md A.1 step 4)
    assert O.mask_counts(0.95, 64, 128, 2) == (60, 61)
    assert O.mask_counts(0.95, 64, 0, 0) == (60, 0)
    assert O.mask_counts(0.8, 0, 50, 2) == (0, 20)
    assert O.mask_counts(0.75, 16, 32, 2) == (12, 12)


def test_tie_free_noise_has_no_ties():
    g = torch.Generator().manual_seed(0)
    n = O.tie_free_noise(512, 192, g, [64, 64, 64])
    for off in (0, 64, 128):
        s = n[:, off:off + 64].sort(dim=-1).values
        assert not (s[:, 1:] == s[:, :-1]).any()


def test_product_vt_load_matches_oracle():
    """m3l_b200.data.vt_load (pure torch, device agnostic) against the oracle restatement of
    utils/pretrain_utils.py:7-57 (itself pinned against the reference in test_oracle_vs_reference.py)."""
    import numpy as np
    import torch
    from m3l_b200.data import vt_load
    from oracle import vtmae_oracle as O
    rng = np.random.default_rng(0)
    for sensors in (1, 2, 4):
        obs = {"image": rng.random((3, 64, 64, 12), dtype=np.float32),
               "tactile": rng.random((3, 3 * sensors * 4, 32, 32), dtype=np.float32) * 2 - 1}
        a = vt_load({k: v.copy() for k, v in obs.items()}, frame_stack=4)
        b = O.vt_load({k: v.copy() for k, v in obs.items()}, frame_stack=4)
        assert sorted(a) == sorted(b)
        for k in a:
            assert torch.equal(torch.as_tensor(a[k]), torch.as_tensor(b[k])), k



@pytest.mark.parametrize("name", VTT_DINO_CASES)
def test_vtt_dino_oracle_matches_reference_golden(name):
    """oracle/vtt_dino_oracle.py against outputs of the unmodified models/VTT.py::VTT frozen by
    oracle/make_golden_vtt_dino.py (runs anywhere: the GPU box has no /root/reference)."""
    from oracle import vtt_dino_oracle as VD
    g = VttDinoGolden(name)
    sd = g.weights()
    for k in sd:
        if sd[k].dtype.is_floating_point and k != "pos_embed.frequency_bands":
            sd[k].requires_grad_(True)
    out = VD.forward_features(sd, g.cfg, g.inputs(), g.masks())
    for k in ("x_norm_regtokens", "x_norm_patchtokens", "x_prenorm"):
        assert torch.equal(out[k].detach(), g.t("out." + k)), k
    g.objective(out).backward()
    for k, has in g.grad_present().items():
        gr = sd[k].grad
        assert (gr is not None and float(gr.abs().max()) > 0) == has, k
    for k, n in g.grad_norms().items():
        if n > 0:
            assert abs(float(sd[k].grad.double().norm()) - n) <= 1e-5 * n, k
    for k, gr in g.full_grads().items():
        assert torch.allclose(sd[k].grad, gr, rtol=1e-5, atol=1e-7), k


def test_product_geometry_matches_oracle_mask_counts():
    """Host logic of the product (engine.make_geometry: the Python-float truncations of pretrain_models.py:223-227 and
    the per-modality rule of reconstruct(), :425,433) against the oracle over a sweep of ratios and token grids."""
    from types import SimpleNamespace
    from m3l_b200 import engine
    from oracle import vtmae_oracle as O
    for n_img, n_tac, nt in ((64, 64, 2), (64, 64, 0), (16, 16, 2), (25, 25, 2), (64, 16, 1), (36, 64, 3)):
        for r in (0.05, 0.3, 0.5, 0.75, 0.8, 0.9, 0.95, 0.99):
            cfg = SimpleNamespace(num_tactiles=nt, n_img=n_img, n_tac=n_tac, masking_ratio=r)
            for use_vision, use_tactile in ((True, True), (True, False), (False, True)):
                if (not use_tactile or nt == 0) and not use_vision:
                    continue
                g = engine.make_geometry(cfg, use_vision, use_tactile)
                ni = n_img if use_vision else 0
                ntt = nt * n_tac if (use_tactile and nt) else 0
                assert (g.nm_img, g.nm_tac) == O.mask_counts(r, ni, ntt, nt), (n_img, n_tac, nt, r, use_vision, use_tactile)
                assert g.n == ni + ntt and g.nv == g.n - g.nm
                gr = engine.make_geometry(cfg, use_vision, use_tactile, reconstruct_ratio=r)
                assert (gr.nm_img, gr.nm_tac) == O.mask_counts_reconstruct(r, ni, ntt, nt)
