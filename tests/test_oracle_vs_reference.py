"""CPU: the oracle (and the product's module layouts) against what the upstream M3L code returns on seeded inputs,
stored under tests/golden/reference/ by oracle/make_golden_reference_checks.py (see there for where the values come
from and how a tensor is stored).  Layouts and pure data movement (vt_load, position tables) are compared exactly.
Computed fp32 results depend on the CPU's summation order (thread count, SIMD width), so against stored values they
get the tolerances of the stored-reference tests in test_oracle_golden.py: losses rtol 1e-6, activations rtol / atol
1e-5; gradients keep rtol 1e-5 / atol 1e-7 and the two-step optimizer trajectory rtol 1e-6 / atol 1e-8."""
import pytest
import torch

from oracle import make_golden_reference_checks as G
from oracle import vtdino_oracle as DO
from oracle import vtmae_oracle as O

LOSS = dict(exact=False, rtol=1e-6)
ACT = dict(exact=False, rtol=1e-5, atol=1e-5)
GRAD = dict(exact=False, rtol=1e-5, atol=1e-7)


def stored(name):
    return G.Stored(G.OUT / f"{name}.npz")


def check(z, key, t, exact=True, rtol=0.0, atol=0.0):
    """t against the stored upstream tensor `key`: shape, the sampled entries, and the sums over all entries."""
    shape, want, (total, mag, nonfinite) = z.tensor(key)
    assert tuple(t.shape) == shape, key
    got = G.sample(t)
    s, m, nf = G.summary(t)
    assert nf == nonfinite, key
    if exact:
        assert torch.isclose(got, want, rtol=0, atol=0, equal_nan=True).all(), key
        assert abs(s - total) <= 1e-12 * mag and abs(m - mag) <= 1e-12 * mag, key
    else:
        assert torch.isclose(got, want, rtol=rtol, atol=atol, equal_nan=True).all(), key
        assert abs(m - mag) <= rtol * mag + atol * t.numel(), key


def assert_weights(z, prefix, sd):
    chk = G.checksum({k: v.detach() for k, v in sd.items()})
    assert abs(chk - z[prefix + "weights_checksum"]) <= 1e-9 * abs(chk), "RNG drift: weights differ"


@pytest.mark.parametrize("ecm,nt,sincos", G.FWD_BWD_CASES)
def test_forward_backward_and_embeddings_match_reference(ecm, nt, sincos):
    z, c = stored("forward_backward"), G.case_key(ecm, nt, sincos) + "/"
    cfg = G.fwd_bwd_cfg(ecm, nt, sincos)
    sd = O.init_state_dict(cfg, seed=3)
    assert_weights(z, c, sd)
    assert G.layout(O.expand_aliases(O.init_state_dict(cfg))) == z[c + "state_dict_layout"]
    for k, v in O.position_buffers(cfg).items():
        check(z, c + "buffer." + k, v)
    x, noise = G.vtmae_batch(cfg, 3, nt, 7)
    for k in O.param_keys(sd):
        sd[k].requires_grad_(True)
    loss = O.vtmae_forward(sd, cfg, x, noise)
    loss.backward()
    check(z, c + "loss", loss, **LOSS)
    for k in O.param_keys(sd):
        if not z[c + "ghas." + k]:
            assert sd[k].grad is None or float(sd[k].grad.abs().max()) == 0.0, k
        else:
            check(z, c + "grad." + k, sd[k].grad, **GRAD)
    with torch.no_grad():
        check(z, c + "embeddings", O.vtmae_embeddings(sd, cfg, x), **ACT)
        if nt:
            check(z, c + "embeddings_vision_only", O.vtmae_embeddings(sd, cfg, x, use_tactile=False), **ACT)


@pytest.mark.parametrize("nt,sincos,ratio,ecm", G.RECONSTRUCT_CASES)
def test_reconstruct_matches_reference(nt, sincos, ratio, ecm):
    """VTMAE.reconstruct (pretrain_models.py:344-586): per-modality mask counts, rec / masked maps, losses."""
    z, c = stored("reconstruct"), G.case_key(nt, sincos, ratio, ecm) + "/"
    cfg = G.reconstruct_cfg(nt, sincos, ecm)
    sd = O.init_state_dict(cfg, seed=5)
    assert_weights(z, c, sd)
    x, noise = G.vtmae_batch(cfg, 3, nt, 11)
    with torch.no_grad():
        mine = O.vtmae_reconstruct(sd, cfg, x, noise, mask_ratio=ratio)
    assert list(mine) == z[c + "keys"]
    for k, v in mine.items():
        check(z, c + k, v, **(LOSS if k.startswith("recon_loss") else ACT))


def test_vt_load_matches_reference():
    z = stored("vt_load")
    a = O.vt_load(G.vt_load_obs(), frame_stack=4)
    assert sorted(a) == z["keys"] == ["image", "tactile1", "tactile2"]
    for k in a:
        check(z, k, a[k])


def test_train_step_matches_reference_optimizer():
    z = stored("train_step")
    cfg = O.VTMAEConfig(depth=1, decoder_depth=1)
    sd = O.init_state_dict(cfg, seed=5)
    assert_weights(z, "", sd)
    x, noise = G.vtmae_batch(cfg, 2, 2, 11)
    st = O.AdamWState()
    for i in range(2):
        lo, _, _ = O.train_step(sd, cfg, x, noise, st)
        check(z, f"loss.{i}", lo, **LOSS)
    for k in O.param_keys(sd):
        check(z, "after." + k, sd[k], exact=False, rtol=1e-6, atol=1e-8)


def test_dino_tac_mae_config_matches_reference():
    """BASELINE.json configs[3], MAE side: 70x70 maps, patch 14, dim 384, tactile-only call (x without 'image':
    pretrain_models.py:148-152), mask 0.8 (train_dino_tac_mae.py:76-80,139-164)."""
    z = stored("dino_tac_mae")
    cfg = G.dino_tac_cfg()
    sd = O.init_state_dict(cfg, seed=9)
    assert_weights(z, "", sd)
    x, noise = G.dino_tac_batch(cfg, 3, 21)
    for k in O.param_keys(sd):
        sd[k].requires_grad_(True)
    loss = O.vtmae_forward(sd, cfg, x, noise)
    loss.backward()
    check(z, "loss", loss, **LOSS)
    for k in O.param_keys(sd):
        if "grad." + k in z:
            check(z, "grad." + k, sd[k].grad, **GRAD)


@pytest.mark.parametrize("regs,with_masks", G.VTT_DINO_CASES)
def test_vtt_dino_forward_features_match_reference(regs, with_masks):
    """models/VTT.py::VTT.forward_features (SURVEY §8 a-16): sinusoidal table, three patch embeddings, shared
    keep-index masks, register tokens, final LayerNorm(eps=1e-6)."""
    from oracle import vtt_dino_oracle as VD
    z, c = stored("vtt_dino"), G.case_key(regs, with_masks) + "/"
    cfg, sd, x, masks = G.vtt_dino_setup(regs, with_masks)
    assert_weights(z, c, sd)
    check(z, c + "pos_table", VD.sinusoidal_table(cfg.pos_grid, cfg.dim))
    out = G.vtt_dino_grads(sd, cfg, x, masks)
    for k in ("x_norm_regtokens", "x_norm_patchtokens", "x_prenorm"):
        check(z, c + "out." + k, out[k], **ACT)
    for k, v in sd.items():
        if not v.requires_grad:
            continue
        if not z[c + "ghas." + k]:
            assert v.grad is None or float(v.grad.abs().max()) == 0.0, k
        else:
            check(z, c + "grad." + k, v.grad, **GRAD)


def test_vtt_dino_product_module_mirrors_reference_state_dict():
    """m3l_b200.vtt.VTT: same state_dict keys / shapes / buffers as models/VTT.py::VTT, same init statistics."""
    from oracle import vtt_dino_oracle as VD
    z = stored("vtt_mirror")
    cfg = VD.VTTDinoConfig(num_register_tokens=1)
    mine = G.product_vtt(cfg, 0, 1)
    b = mine.state_dict()
    assert G.layout(b) == z["state_dict_layout"]
    check(z, "frequency_bands", b["pos_embed.frequency_bands"])
    check(z, "pos_embed", mine.pos_embed(torch.device("cpu")))
    w = b["transformer.layers.0.1.net.1.weight"]
    assert abs(float(w.std()) - 0.02) < 2e-3 and float(b["transformer.layers.0.1.net.1.bias"].abs().max()) == 0.0
    dtypes = {str(getattr(torch, n)): getattr(torch, n) for n in ("float32", "float64", "int64", "bool")}
    mine.load_state_dict({k: torch.zeros(s, dtype=dtypes[d]) for k, s, d in z["state_dict_layout"]})


def test_dino_head_loss_and_ema_match_reference_files():
    """oracle/vtdino_oracle.py against tactile_ssl/model/layers/dino_head.py, tactile_ssl/loss/dino_loss.py and
    tactile_ssl/utils/ema.py: head output, two rounds of centred teacher softmax / centre EMA / loss, parameter EMA."""
    z = stored("dino_head_loss_ema")
    head, x, t_out, s_list, lin_a, lin_b = G.dino_head_setup()
    check(z, "head_out", DO.dino_head_forward(head, x), **ACT)
    for i, (t_soft, center, loss) in enumerate(G.dino_center_steps(t_out, s_list)):
        check(z, f"t_soft.{i}", t_soft, **ACT)
        check(z, f"center.{i}", center, **ACT)
        check(z, f"loss.{i}", loss, **LOSS)
    for j, (pa, pb) in enumerate(zip(lin_a, lin_b)):
        check(z, f"ema.{j}", DO.ema(pa, pb, 0.97), **ACT)


def test_sb3_checkpoint_round_trip_with_the_reference_extractor(tmp_path):
    """SB3's CheckpointCallback (utils/callbacks.py:126-133 -> BaseAlgorithm.save) writes a zip whose `policy.pth`
    member is torch.save(policy.state_dict()); the MAE part of a policy lives under `features_extractor.`.  A
    checkpoint laid out as the upstream MAEExtractor's loads strictly into the product extractor, and one written from
    the product has exactly the upstream layout: saved policies stay interchangeable."""
    z = stored("sb3_policy")
    mine = G.mae_extractor_policy()
    assert G.layout(mine.state_dict()) == z["policy_layout"]
    theirs = {k: v + 0.5 for k, v in mine.state_dict().items()}      # shared modules appear under two keys: equal values
    # upstream layout -> zip -> product
    G.save_sb3_zip(theirs, tmp_path / "ref.zip")
    sd = G.load_policy_pth(tmp_path / "ref.zip")
    assert set(sd) == set(mine.state_dict())
    mine.load_state_dict(sd, strict=True)
    for k, v in theirs.items():
        assert torch.equal(mine.state_dict()[k], v), k
    # product -> zip -> upstream layout
    with torch.no_grad():
        for p in mine.parameters():
            p.mul_(1.01)
    G.save_sb3_zip(mine.state_dict(), tmp_path / "mine.zip")
    back = G.load_policy_pth(tmp_path / "mine.zip")
    assert G.layout(back) == z["policy_layout"]
    for k, v in mine.state_dict().items():
        assert torch.equal(back[k], v), k
