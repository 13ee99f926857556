"""TEST INFRASTRUCTURE - the stored upstream side of tests/test_oracle_vs_reference.py.

Those tests compare the oracle with the upstream M3L code (models/pretrain_models.py, models/VTT.py,
tactile_ssl/...) on seeded inputs.  The upstream tree is not part of this repository, so what its side returned is
stored under tests/golden/reference/ (one file per test) and the tests compare against that:

    python -m oracle.make_golden_reference_checks

The stored values are computed by the oracle (and, for state_dict layouts, the product modules) that these same
comparisons held equal to the upstream code, bit-for-bit (torch.equal) for outputs and losses, to rtol 1e-5 for
gradients and 1e-6 for optimizer trajectories, so on these inputs they are the upstream results.  Inputs and weights
are re-derived from their seeds by the builders below (a stored checksum detects RNG drift).  A tensor is stored as
its shape, a fixed sample of N_SAMPLE entries, and float64 sums over all entries (summary()): small
enough to keep every file far below 1 MB.
"""
from __future__ import annotations

import io
import json
import sys
import zipfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import vtdino_oracle as DO  # noqa: E402
from oracle import vtmae_oracle as O  # noqa: E402
from oracle import vtt_dino_oracle as VD  # noqa: E402

OUT = ROOT / "tests" / "golden" / "reference"
N_SAMPLE = 16

FWD_BWD_CASES = [(False, 2, True), (False, 0, True), (True, 2, True), (False, 2, False)]          # ecm, nt, sincos
RECONSTRUCT_CASES = [(2, True, None, False), (2, False, 0.5, False), (0, True, 0.8, False), (2, True, 0.6, True)]
VTT_DINO_CASES = [(1, False), (1, True), (0, False), (2, True)]                                   # regs, with_masks


def case_key(*params) -> str:
    return "_".join(str(p) for p in params)


# ------------------------------------------------------------------------------------------------ storage format
def _idx(numel: int) -> torch.Tensor:
    return torch.linspace(0, numel - 1, min(N_SAMPLE, numel), dtype=torch.float64).round().long()


class Store:
    """One file per test: `index` (JSON: plain values, and per tensor its shape and where its entries sit),
    `samples` (float32: the sampled entries of every tensor) and `stats` (float64: summary(), three per tensor)."""

    def __init__(self):
        self.index, self.samples, self.stats = {}, [], []

    def __setitem__(self, key, value):               # plain JSON value: checksums, flags, key lists, layouts
        self.index[key] = value

    def put(self, key: str, t) -> None:
        t = torch.as_tensor(t).detach()
        f = t.reshape(-1).float()
        at = sum(len(a) for a in self.samples)
        self.samples.append(f[_idx(f.numel())].numpy().copy())
        self.index[key] = {"shape": list(t.shape), "at": at, "n": len(self.samples[-1]), "stat": len(self.stats) // 3}
        self.stats += summary(t)

    def save(self, path: Path) -> None:
        np.savez_compressed(path, index=np.frombuffer(json.dumps(self.index).encode(), dtype=np.uint8),
                            samples=np.concatenate(self.samples or [np.zeros(0, np.float32)]),
                            stats=np.array(self.stats, dtype=np.float64))


class Stored:
    """Reader of a Store file: z[key] is the plain value, z.tensor(key) -> (shape, sampled entries, summary)."""

    def __init__(self, path: Path):
        z = np.load(path)
        self.index = json.loads(bytes(z["index"]).decode())
        self.samples, self.stats = torch.from_numpy(z["samples"]), z["stats"]

    def __getitem__(self, key):
        return self.index[key]

    def __contains__(self, key):
        return key in self.index

    def tensor(self, key):
        e = self.index[key]
        i = 3 * e["stat"]
        return tuple(e["shape"]), self.samples[e["at"]:e["at"] + e["n"]], [float(v) for v in self.stats[i:i + 3]]


def sample(t) -> torch.Tensor:
    f = torch.as_tensor(t).detach().reshape(-1).float()
    return f[_idx(f.numel())]


def summary(t) -> list:
    """[sum, sum of magnitudes] of the finite entries, and sum over the others of (position + 1) * (1 for +inf,
    2 for -inf, 3 for nan): masked maps mark masked patches with non-finite values."""
    f = torch.as_tensor(t).detach().reshape(-1).double()
    fin = torch.isfinite(f)
    code = torch.where(torch.isnan(f), 3.0, torch.where(f > 0, 1.0, 2.0))
    pos = torch.arange(1, f.numel() + 1, dtype=torch.float64)
    return [float(f[fin].sum()), float(f[fin].abs().sum()), float((pos * code)[~fin].sum())]


def checksum(sd) -> float:
    return float(sum(v.double().abs().sum() for k, v in sorted(sd.items())))


# ------------------------------------------------------------------------------------------------ seeded builders
def vtmae_batch(cfg, B, nt, seed):
    g = torch.Generator().manual_seed(seed)
    x = {"image": torch.rand(B, 12, 64, 64, generator=g)}
    for i in range(nt):
        x[f"tactile{i + 1}"] = torch.rand(B, 12, 32, 32, generator=g)
    return x, O.tie_free_noise(B, cfg.n_img + nt * cfg.n_tac, g, [64] * (1 + nt))


def fwd_bwd_cfg(ecm, nt, sincos):
    return O.VTMAEConfig(early_conv_masking=ecm, num_tactiles=nt, use_sincosmod_encodings=sincos, depth=2, decoder_depth=1)


def reconstruct_cfg(nt, sincos, ecm):
    return O.VTMAEConfig(num_tactiles=nt, use_sincosmod_encodings=sincos, depth=2, decoder_depth=1, early_conv_masking=ecm)


def dino_tac_cfg():
    return O.VTMAEConfig(image_size=(70, 70), tactile_size=(70, 70), image_patch_size=14, tactile_patch_size=14, dim=384,
                         depth=2, heads=4, mlp_dim=768, decoder_dim=384, decoder_depth=1, decoder_heads=4, masking_ratio=0.8)


def dino_tac_batch(cfg, B, seed):
    """Tactile-only call (x without 'image'): two 70 x 70 maps and their mask noise."""
    g = torch.Generator().manual_seed(seed)
    x = {f"tactile{i + 1}": torch.rand(B, 12, 70, 70, generator=g) for i in range(2)}
    return x, O.tie_free_noise(B, 2 * cfg.n_tac, g, [cfg.n_tac] * 2)


def vt_load_obs():
    rng = np.random.default_rng(0)
    return {"image": rng.random((2, 64, 64, 12), dtype=np.float32),
            "tactile": (rng.random((2, 24, 32, 32), dtype=np.float32) * 2 - 1)}


def product_vtt(cfg, seed, regs):
    """m3l_b200.vtt.VTT, the drop-in for models/VTT.py::VTT (same state_dict layout and init statistics)."""
    from m3l_b200.vtt import VTT
    torch.manual_seed(seed)
    return VTT(image_size=cfg.image_size, tactile_size=cfg.tactile_size, image_patch_size=cfg.image_patch_size,
               tactile_patch_size=cfg.tactile_patch_size, dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, mlp_dim=cfg.mlp_dim,
               num_tactiles=cfg.num_tactiles, image_channels=cfg.image_channels, tactile_channels=cfg.tactile_channels,
               dim_head=cfg.dim_head, num_register_tokens=regs, pos_embed_fn="sinusoidal")


def vtt_dino_setup(regs, with_masks):
    """Weights (register tokens drawn at std 0.5 so that they matter), inputs and keep-index masks."""
    cfg = VD.VTTDinoConfig(depth=2, num_register_tokens=regs)
    sd = {k: v.clone() for k, v in product_vtt(cfg, 13, regs).state_dict().items()}
    if regs:
        sd["register_tokens"] = torch.empty_like(sd["register_tokens"]).normal_(0, 0.5)
    g = torch.Generator().manual_seed(3)
    B = 3
    x = {"image": torch.rand(B, 12, 64, 64, generator=g), "tactile1": torch.rand(B, 12, 32, 32, generator=g),
         "tactile2": torch.rand(B, 12, 32, 32, generator=g)}
    masks = [torch.stack([torch.randperm(64, generator=g)[:k] for _ in range(B)]) for k in (40, 40)] if with_masks else None
    for k in sd:
        if sd[k].dtype.is_floating_point and k != "pos_embed.frequency_bands":
            sd[k].requires_grad_(True)
    return cfg, sd, x, masks


def vtt_dino_grads(sd, cfg, x, masks):
    """Forward, then the gradient of sum(patch tokens of a second forward) + sum(register tokens of the first ^ 2)."""
    out = VD.forward_features(sd, cfg, x, masks)
    (VD.forward_features(sd, cfg, x, masks)["x_norm_patchtokens"].sum() + (out["x_norm_regtokens"] ** 2).sum()).backward()
    return out


def dino_head_setup():
    """DINOHead(in_dim=64, out_dim=96, hidden_dim=128, bottleneck_dim=32) weights, its input, teacher / student outputs."""
    g = torch.Generator().manual_seed(0)
    shapes = {"mlp.0.weight": (128, 64), "mlp.0.bias": (128,), "mlp.2.weight": (128, 128), "mlp.2.bias": (128,),
              "mlp.4.weight": (32, 128), "mlp.4.bias": (32,), "last_layer.weight_g": (96, 1), "last_layer.weight_v": (96, 32)}
    head = {k: torch.randn(*s, generator=g) * (0.02 if k.endswith("weight") else 0.1) for k, s in shapes.items()}
    head["last_layer.weight_g"] = 1 + 0.1 * torch.randn(96, 1, generator=g)
    x = torch.randn(5, 3, 64, generator=g)
    t_out = torch.randn(10, 1, 96, generator=g)
    s_list = [torch.randn(5, 1, 96, generator=g) for _ in range(3)]
    lin_a = [torch.randn(5, 7, generator=g), torch.randn(5, generator=g)]
    lin_b = [torch.randn(5, 7, generator=g), torch.randn(5, generator=g)]
    return head, x, t_out, s_list, lin_a, lin_b


def dino_center_steps(t_out, s_list):
    """Two rounds of DINOLoss: centred teacher softmax, centre EMA, cross-entropy over the student crops."""
    center = torch.zeros(1, 96)
    rounds = []
    for _ in range(2):
        t_soft = DO.softmax_center_teacher(t_out, center, 0.05)
        center = DO.center_update(center, t_out)
        rounds.append((t_soft, center, DO.dino_loss(s_list, list(t_soft.view(2, -1, 1, 96)))))
    return rounds


def mae_extractor_policy(seed_model=1, seed_ext=2):
    """The slice of an SB3 ActorCriticPolicy that holds the MAE: features_extractor (MAEExtractor) + an action head."""
    from m3l_b200 import VTT, VTMAE, MAEExtractor
    cfg = O.VTMAEConfig(depth=2, decoder_depth=1)
    torch.manual_seed(seed_model)
    enc = VTT(image_size=cfg.image_size, tactile_size=cfg.tactile_size, image_patch_size=cfg.image_patch_size,
              tactile_patch_size=cfg.tactile_patch_size, dim=cfg.dim, depth=cfg.depth, heads=cfg.heads, mlp_dim=cfg.mlp_dim,
              num_tactiles=cfg.num_tactiles, image_channels=cfg.image_channels, tactile_channels=cfg.tactile_channels,
              frame_stack=cfg.frame_stack)
    mae = VTMAE(encoder=enc, decoder_dim=cfg.decoder_dim, masking_ratio=cfg.masking_ratio, decoder_depth=cfg.decoder_depth,
                decoder_heads=cfg.decoder_heads, num_tactiles=cfg.num_tactiles, frame_stack=cfg.frame_stack)
    torch.manual_seed(seed_ext)

    class Policy(torch.nn.Module):
        def __init__(self, ext):
            super().__init__()
            self.features_extractor = ext
            self.action_net = torch.nn.Linear(cfg.dim, 4)

    return Policy(MAEExtractor(None, mae, cfg.dim, False, cfg.frame_stack))


def save_sb3_zip(policy_state, path):
    """What SB3's BaseAlgorithm.save writes: a zip whose `policy.pth` member is torch.save(policy.state_dict())."""
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", "{}")
        for member, obj in (("policy.pth", policy_state), ("policy.optimizer.pth", {}), ("pytorch_variables.pth", {})):
            buf = io.BytesIO()
            torch.save(obj, buf)
            z.writestr(member, buf.getvalue())
        z.writestr("_stable_baselines3_version", "2.1.0")


def load_policy_pth(path):
    with zipfile.ZipFile(path) as z:
        return torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu")


def layout(sd) -> list:
    return [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()]


# ------------------------------------------------------------------------------------------------ generators
def gen_forward_backward(out):
    for ecm, nt, sincos in FWD_BWD_CASES:
        c = case_key(ecm, nt, sincos)
        cfg = fwd_bwd_cfg(ecm, nt, sincos)
        sd = O.init_state_dict(cfg, seed=3)
        out[c + "/weights_checksum"] = checksum(sd)
        out[c + "/state_dict_layout"] = layout(O.expand_aliases(sd))
        for k, v in O.position_buffers(cfg).items():
            out.put(c + "/buffer." + k, v)
        x, noise = vtmae_batch(cfg, 3, nt, 7)
        for k in O.param_keys(sd):
            sd[k].requires_grad_(True)
        loss = O.vtmae_forward(sd, cfg, x, noise)
        loss.backward()
        out.put(c + "/loss", loss)
        for k in O.param_keys(sd):
            out[c + "/ghas." + k] = bool(sd[k].grad is not None)
            if sd[k].grad is not None:
                out.put(c + "/grad." + k, sd[k].grad)
        with torch.no_grad():
            out.put(c + "/embeddings", O.vtmae_embeddings(sd, cfg, x))
            if nt:
                out.put(c + "/embeddings_vision_only", O.vtmae_embeddings(sd, cfg, x, use_tactile=False))


def gen_reconstruct(out):
    for nt, sincos, ratio, ecm in RECONSTRUCT_CASES:
        c = case_key(nt, sincos, ratio, ecm)
        cfg = reconstruct_cfg(nt, sincos, ecm)
        sd = O.init_state_dict(cfg, seed=5)
        out[c + "/weights_checksum"] = checksum(sd)
        x, noise = vtmae_batch(cfg, 3, nt, 11)
        with torch.no_grad():
            rec = O.vtmae_reconstruct(sd, cfg, x, noise, mask_ratio=ratio)
        out[c + "/keys"] = list(rec)
        for k, v in rec.items():
            out.put(c + "/" + k, v)


def gen_vt_load(out):
    res = O.vt_load(vt_load_obs(), frame_stack=4)
    out["keys"] = sorted(res)
    for k, v in res.items():
        out.put(k, v)


def gen_train_step(out):
    cfg = O.VTMAEConfig(depth=1, decoder_depth=1)
    sd = O.init_state_dict(cfg, seed=5)
    out["weights_checksum"] = checksum(sd)
    x, noise = vtmae_batch(cfg, 2, 2, 11)
    st = O.AdamWState()
    for i in range(2):
        lo, _, _ = O.train_step(sd, cfg, x, noise, st)
        out.put(f"loss.{i}", lo)
    for k in O.param_keys(sd):
        out.put("after." + k, sd[k])


def gen_dino_tac(out):
    cfg = dino_tac_cfg()
    sd = O.init_state_dict(cfg, seed=9)
    out["weights_checksum"] = checksum(sd)
    x, noise = dino_tac_batch(cfg, 3, 21)
    for k in O.param_keys(sd):
        sd[k].requires_grad_(True)
    loss = O.vtmae_forward(sd, cfg, x, noise)
    loss.backward()
    out.put("loss", loss)
    for k in O.param_keys(sd):
        if sd[k].grad is not None:
            out.put("grad." + k, sd[k].grad)


def gen_vtt_dino(out):
    for regs, with_masks in VTT_DINO_CASES:
        c = case_key(regs, with_masks)
        cfg, sd, x, masks = vtt_dino_setup(regs, with_masks)
        out[c + "/weights_checksum"] = checksum({k: v.detach() for k, v in sd.items()})
        out.put(c + "/pos_table", VD.sinusoidal_table(cfg.pos_grid, cfg.dim))
        res = vtt_dino_grads(sd, cfg, x, masks)
        for k in ("x_norm_regtokens", "x_norm_patchtokens", "x_prenorm"):
            out.put(c + "/out." + k, res[k])
        for k, v in sd.items():
            if v.requires_grad:
                out[c + "/ghas." + k] = bool(v.grad is not None and float(v.grad.abs().max()) > 0)
                if v.grad is not None:
                    out.put(c + "/grad." + k, v.grad)


def gen_vtt_mirror(out):
    cfg = VD.VTTDinoConfig(num_register_tokens=1)
    m = product_vtt(cfg, 0, 1)
    out["state_dict_layout"] = layout(m.state_dict())
    out.put("frequency_bands", m.state_dict()["pos_embed.frequency_bands"])
    out.put("pos_embed", m.pos_embed(torch.device("cpu")))


def gen_dino_head(out):
    head, x, t_out, s_list, lin_a, lin_b = dino_head_setup()
    out.put("head_out", DO.dino_head_forward(head, x))
    for i, (t_soft, center, loss) in enumerate(dino_center_steps(t_out, s_list)):
        out.put(f"t_soft.{i}", t_soft)
        out.put(f"center.{i}", center)
        out.put(f"loss.{i}", loss)
    for j, (pa, pb) in enumerate(zip(lin_a, lin_b)):
        out.put(f"ema.{j}", DO.ema(pa, pb, 0.97))


def gen_sb3(out):
    out["policy_layout"] = layout(mae_extractor_policy().state_dict())


GENERATORS = {
    "forward_backward": gen_forward_backward, "reconstruct": gen_reconstruct, "vt_load": gen_vt_load,
    "train_step": gen_train_step, "dino_tac_mae": gen_dino_tac, "vtt_dino": gen_vtt_dino, "vtt_mirror": gen_vtt_mirror,
    "dino_head_loss_ema": gen_dino_head, "sb3_policy": gen_sb3,
}


def main():
    torch.set_num_threads(8)
    OUT.mkdir(parents=True, exist_ok=True)
    for name, fn in GENERATORS.items():
        out = Store()
        fn(out)
        out.save(OUT / f"{name}.npz")
        print(f"{name}: {(OUT / (name + '.npz')).stat().st_size / 1e3:.1f} kB")


if __name__ == "__main__":
    main()
