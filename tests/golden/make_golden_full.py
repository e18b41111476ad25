"""Full-size golden fixtures from the UNMODIFIED reference (run in the build container only; ~5 min of CPU).

    python tests/golden/make_golden_full.py       # needs /root/reference; writes tests/golden/full_traj.npz

Same import recipe as make_golden.py (reference modules from /root/reference/src, NAC stubbed).  Cases, all with the
repo-default model (H = 768, L = 5, 1 head, time 256), diffusion_steps = 50, weights oracle.make_state_dict(seed 0):

  c1_traj   BASELINE C1/C2 utterance: B = 1, T = 750, S = 64, the full 50-step CFG sampling loop (w = 3, unconditional =
            zero text): guided eps_hat of the first and the last step and the final latent
  c3_fwd    BASELINE C3 utterance: T = 2250, S = 192, one forward, all 5 layers (t = 17)
  c5_u{0,1,2}  three speech-length-predictor-sized utterances of BASELINE C5 (2 s / 11 s / 20 s -> T = 150 / 825 / 1500,
            S = 13 / 70 / 128): each sampled ON ITS OWN (the reference has no masks: per-utterance, unpadded), 50-step CFG

Inputs regenerate bit-identically from the seeds (oracle.make_inputs), so only OUTPUTS are stored, sub-sampled along the
frame axis (every `stride`-th frame, all 768 channels) plus the float64 norm of the full tensor.
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from make_golden import build_reference, import_reference, reference_sampler  # noqa: E402
from oracle import ditto_oracle as O  # noqa: E402

STRIDE = 50   # keeps the file under 1 MB
W = 3.0
STEPS = 50
# name, input seed, T, S
TRAJ_CASES = [("c1_traj", 11, 750, 64), ("c5_u0", 12, 150, 13), ("c5_u1", 13, 825, 70), ("c5_u2", 14, 1500, 128)]


def cfg_trajectory(ref, gen, c, x, text, noise):
    xs = x.clone()
    first = last = None
    norms = []
    with torch.no_grad():
        for t_val in reversed(range(c.diffusion_steps)):
            tt = torch.full((x.shape[0],), t_val, dtype=torch.long)
            e_c = ref(xs, text, tt)                                   # reference DiTTO.forward (DiTTO.py:66-94)
            e_u = ref(xs, torch.zeros_like(text), tt)
            eps = e_u + W * (e_c - e_u)                               # CFG extension
            xs = O.p_sample_update(xs, eps, noise[t_val], tt, gen.betas, gen.alphas, gen.alphas_cumprod)  # SpeechGenerator.py:137-147
            norms.append(float(eps.double().norm()))
            if t_val == c.diffusion_steps - 1:
                first = eps.clone()
            if t_val == 0:
                last = eps.clone()
    return first, last, xs, norms


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    M, SG = import_reference()
    c = O.OracleConfig(768, 5, 1, 256, 768, STEPS)
    sd = O.make_state_dict(c, seed=0)
    ref = build_reference(M, c, sd)
    gen = reference_sampler(SG, ref, c)
    out = {"meta": np.array([c.hidden_dim, c.num_layers, c.num_heads, c.time_dim, c.text_dim, c.diffusion_steps, 0, STRIDE]),
           "w": np.array([W])}
    for name, seed, T, S in TRAJ_CASES:
        t0 = time.time()
        x, text, noise = O.make_inputs(1, T, S, c, seed=seed, steps_noise=STEPS)
        first, last, final, norms = cfg_trajectory(ref, gen, c, x, text, noise)
        out[f"{name}::shape"] = np.array([seed, T, S])
        out[f"{name}::eps_first_sub"] = first[:, ::STRIDE].numpy()
        out[f"{name}::eps_last_sub"] = last[:, ::STRIDE].numpy()
        out[f"{name}::final_sub"] = final[:, ::STRIDE].numpy()
        out[f"{name}::norms"] = np.array([float(first.double().norm()), float(last.double().norm()), float(final.double().norm())])
        out[f"{name}::eps_norms"] = np.array(norms)
        print(f"{name}: T={T} S={S} |final|={float(final.norm()):.4e} ({time.time() - t0:.0f} s)", flush=True)
    # C3: one forward at T = 2250, S = 192, all five layers
    x, text, _ = O.make_inputs(1, 2250, 192, c, seed=15)
    t = torch.tensor([17], dtype=torch.long)
    with torch.no_grad():
        o = ref(x, text, t)
    out["c3_fwd::shape"] = np.array([15, 2250, 192, 17])
    out["c3_fwd::out_sub"] = o[:, ::STRIDE].numpy()
    out["c3_fwd::norms"] = np.array([float(o.double().norm())])
    print("c3_fwd: |out| =", float(o.norm()), flush=True)
    np.savez_compressed(os.path.join(HERE, "full_traj.npz"), **out)
    print("full_traj.npz written,", os.path.getsize(os.path.join(HERE, "full_traj.npz")) / 1e6, "MB")


if __name__ == "__main__":
    main()
