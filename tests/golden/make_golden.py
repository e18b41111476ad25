"""Mint golden fixtures from the UNMODIFIED reference (run in the build container only).

    python tests/golden/make_golden.py            # needs /root/reference; writes tests/golden/*.npz

The reference modules are imported from /root/reference/src exactly as they are:
  * model.DiTTO.DiTTO            (src/model/DiTTO.py)      -- NAC replaced by a stub, SURVEY.md appendix B
  * components.DiT.*             (src/components/DiT.py)
  * model.SpeechGenerator.SpeechGenerator.__p_sample  (src/model/SpeechGenerator.py:131-147) -- the class is
    imported with the un-vendored ``bigvgan_v2_24khz_100band_256x`` package stubbed in sys.modules and is
    instantiated with object.__new__ (its __init__ downloads checkpoints); only __p_sample and the schedule
    lines :70-72 are exercised.
Weights come from oracle.make_state_dict (seeded, CPU) and are loaded with load_state_dict, inputs from
oracle.make_inputs; both regenerate bit-identically on the GPU box, so the large-config fixtures only
store (sub-sampled) reference OUTPUTS.  The tiny config stores everything, weights included.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF_SRC = "/root/reference/src"

from oracle import ditto_oracle as O  # noqa: E402


class _StubNAC(nn.Module):
    def __init__(self, **kw):
        super().__init__()
        self.language_model = nn.Identity()
        self.audio_encoder = nn.Identity()

    def load_state_dict(self, *a, **k):  # noqa: D401
        return None


def import_reference():
    sys.path.insert(0, REF_SRC)
    pkg = types.ModuleType("bigvgan_v2_24khz_100band_256x")
    pkg.bigvgan = types.ModuleType("bigvgan_v2_24khz_100band_256x.bigvgan")
    mel = types.ModuleType("bigvgan_v2_24khz_100band_256x.meldataset")
    mel.get_mel_spectrogram = None
    sys.modules["bigvgan_v2_24khz_100band_256x"] = pkg
    sys.modules["bigvgan_v2_24khz_100band_256x.bigvgan"] = pkg.bigvgan
    sys.modules["bigvgan_v2_24khz_100band_256x.meldataset"] = mel
    import model.DiTTO as M
    M.NAC = _StubNAC
    import model.SpeechGenerator as SG
    return M, SG


def build_reference(M, cfg: O.OracleConfig, sd):
    real_load = torch.load
    torch.load = lambda *a, **k: {"model_state_dict": {}}
    try:
        ref = M.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=cfg.num_heads,
                      time_dim=cfg.time_dim, text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps,
                      nac_model_path="unused").eval()
    finally:
        torch.load = real_load
    missing, unexpected = ref.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all(k.startswith("nac.") for k in missing), missing
    return ref


def reference_sampler(SG, ref, cfg):
    """A SpeechGenerator shell carrying just what __p_sample reads (SpeechGenerator.py:70-72,131-147)."""
    gen = object.__new__(SG.SpeechGenerator)
    gen.device = "cpu"
    gen.ditto_model = ref
    gen.betas = ref.cosine_beta_schedule(cfg.diffusion_steps)
    gen.alphas = 1.0 - gen.betas
    gen.alphas_cumprod = torch.cumprod(gen.alphas, dim=0)
    return gen


def block_taps(ref, x, text, t):
    taps = {}
    hooks = [blk.register_forward_hook(lambda m, i, o, k=k: taps.__setitem__(f"block{k}", o.detach().clone()))
             for k, blk in enumerate(ref.blocks)]
    hooks.append(ref.ada_ln.register_forward_hook(lambda m, i, o: taps.__setitem__("adaln", o.detach().clone())))
    with torch.no_grad():
        out = ref(x, text, t)
    for h in hooks:
        h.remove()
    return out, taps


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    M, SG = import_reference()

    # ---------------- tiny config: everything stored ----------------
    cfg = O.OracleConfig(hidden_dim=64, num_layers=2, num_heads=2, time_dim=32, text_dim=64, diffusion_steps=8)
    sd = O.make_state_dict(cfg, seed=3)
    ref = build_reference(M, cfg, sd)
    B, T, S = 2, 24, 8
    x, text, noise = O.make_inputs(B, T, S, cfg, seed=4, steps_noise=cfg.diffusion_steps)
    t = torch.tensor([5, 2], dtype=torch.long)
    out, taps = block_taps(ref, x, text, t)
    # reference sampler, no guidance: the loop of SpeechGenerator.py:161-163 with seeded randn_like
    gen = reference_sampler(SG, ref, cfg)
    xs = x.clone()
    p_sample = gen._SpeechGenerator__p_sample
    ref_noise = torch.empty_like(noise)
    for t_val in reversed(range(cfg.diffusion_steps)):
        tt = torch.full((B,), t_val, dtype=torch.long)
        torch.manual_seed(1000 + t_val)
        ref_noise[t_val] = torch.randn_like(xs)         # what __p_sample will draw (eval mode: no other RNG use)
        torch.manual_seed(1000 + t_val)
        xs = p_sample(xs, tt, text)
    # q_sample with the betas-as-alphas_cumprod quirk (DiTTO.py:106-126)
    qs = ref.q_sample(x, t, noise[0])
    rot = ref.rotary(T, "cpu")
    arrays = {f"sd::{k}": v.numpy() for k, v in sd.items()}
    arrays.update(x=x.numpy(), text=text.numpy(), t=t.numpy(), out=out.numpy(), ref_noise=ref_noise.numpy(),
                  sampled=xs.numpy(), q_sample=qs.numpy(), q_noise=noise[0].numpy(), rotary=rot.numpy(),
                  betas=gen.betas.numpy(), alphas=gen.alphas.numpy(), alphas_cumprod=gen.alphas_cumprod.numpy(),
                  cfg=np.array([cfg.hidden_dim, cfg.num_layers, cfg.num_heads, cfg.time_dim, cfg.text_dim,
                                cfg.diffusion_steps]))
    arrays.update({f"tap::{k}": v.numpy() for k, v in taps.items()})
    np.savez_compressed(os.path.join(HERE, "tiny_full.npz"), **arrays)
    print("tiny_full.npz written; |out| =", float(out.norm()))

    # ---------------- schedules (known-answer vectors quoted in SURVEY.md 8a11) ----------------
    sch = {}
    for steps in (50, 1000):
        b = ref.cosine_beta_schedule(steps)
        a = 1.0 - b
        sch[f"betas{steps}"] = b.numpy()
        sch[f"alphas_cumprod{steps}"] = torch.cumprod(a, 0).numpy()
    np.savez_compressed(os.path.join(HERE, "schedules.npz"), **sch)

    # ---------------- full-size configs: seeded weights, sub-sampled reference outputs ----------------
    full = {}
    cases = [
        # name, cfg, weight seed, input seed, B, T, S, t
        ("c1_default", O.OracleConfig(768, 5, 1, 256, 768, 50), 0, 1, 1, 750, 64, [37]),
        ("ctor_default", O.OracleConfig(768, 12, 12, 256, 768, 50), 0, 1, 1, 200, 32, [11]),
        ("ragged", O.OracleConfig(768, 5, 1, 256, 768, 50), 0, 2, 2, 173, 19, [49, 0]),
    ]
    for name, c, wseed, iseed, B, T, S, tv in cases:
        sd = O.make_state_dict(c, seed=wseed)
        ref = build_reference(M, c, sd)
        x, text, _ = O.make_inputs(B, T, S, c, seed=iseed)
        t = torch.tensor(tv, dtype=torch.long)
        out, taps = block_taps(ref, x, text, t)
        stride = 16   # keeps the file under 1 MB
        full[f"{name}::meta"] = np.array([c.hidden_dim, c.num_layers, c.num_heads, c.time_dim, c.text_dim,
                                          c.diffusion_steps, wseed, iseed, B, T, S, stride])
        full[f"{name}::t"] = t.numpy()
        full[f"{name}::out_sub"] = out[:, ::stride].numpy()
        full[f"{name}::out_norm"] = np.array([float(out.double().norm())])
        full[f"{name}::adaln_sub"] = taps["adaln"][:, ::stride].numpy()
        full[f"{name}::block0_sub"] = taps["block0"][:, ::stride].numpy()
        print(name, "done; |out| =", float(out.norm()))
    np.savez_compressed(os.path.join(HERE, "full_size.npz"), **full)

    # ---------------- 50-step CFG trajectory, small T, default model (reference forward x2 per step) ------------
    c = O.OracleConfig(768, 5, 1, 256, 768, 50)
    sd = O.make_state_dict(c, seed=0)
    ref = build_reference(M, c, sd)
    gen = reference_sampler(SG, ref, c)
    B, T, S, w = 2, 96, 24, 3.0
    x, text, noise = O.make_inputs(B, T, S, c, seed=7, steps_noise=c.diffusion_steps)
    xs = x.clone()
    eps_norms, eps_first, eps_last = [], None, None
    with torch.no_grad():
        for t_val in reversed(range(c.diffusion_steps)):
            tt = torch.full((B,), t_val, dtype=torch.long)
            e_c = ref(xs, text, tt)
            e_u = ref(xs, torch.zeros_like(text), tt)
            eps = e_u + w * (e_c - e_u)                       # the CFG extension (not reference code)
            # the update with the reference's own formula object: reuse __p_sample's arithmetic by
            # restating it on gen's tables (SpeechGenerator.py:137-147)
            xs = O.p_sample_update(xs, eps, noise[t_val], tt, gen.betas, gen.alphas, gen.alphas_cumprod)
            eps_norms.append(float(eps.double().norm()))
            if t_val == c.diffusion_steps - 1:
                eps_first = eps.clone()
            if t_val == 0:
                eps_last = eps.clone()
    stride = 2   # every other frame keeps the file under 1 MB; the norm of the full final latent is stored beside it
    np.savez_compressed(os.path.join(HERE, "cfg_traj.npz"),
                        meta=np.array([B, T, S, 7, 0, c.diffusion_steps]), w=np.array([w]), stride=np.array([stride]),
                        eps_norms=np.array(eps_norms), eps_first=eps_first[:, ::stride].numpy(),
                        eps_last=eps_last[:, ::stride].numpy(), final=xs[:, ::stride].numpy(),
                        final_norm=np.array([float(xs.double().norm())]))
    print("cfg_traj.npz written; |final| =", float(xs.norm()))


if __name__ == "__main__":
    main()
