"""Noise schedules and per-step update coefficients for the sampler variants (SURVEY.md 8f row 4).

The reference knows one sampler: DDPM ancestral sampling with sigma_t^2 = beta_t over every one of
``ConfigDiTTO.DIFFUSION_STEPS`` timesteps of the cosine schedule (src/model/SpeechGenerator.py:70-72,131-164;
src/model/DiTTO.py:96-104).  Its update has the form

    x_prev = c1 (x - c2 eps) + c3 z                                     (SpeechGenerator.py:143-145)

and so do DDIM(eta) and DDPM over a sub-sequence of the timesteps, only with other (c1, c2, c3).  The device kernel
(``cfg_update_kernel``) reads the three numbers from a ``[diffusion_steps, 3]`` table indexed by the model timestep;
this module builds such tables on the host in float64 (they are a few hundred scalars) and
``ditto_engine_load_update_table`` hands them to the engine.  Nothing here touches the hot path.

Variants (all extensions -- the reference has none of them; the DiTTo-TTS paper's inference setting is 25 steps,
CFG scale 5.0, noise-schedule scale-shift 0.3, PDF p.25 Fig. 6):
  * ``spaced_timesteps``      -- K of the model's timesteps, descending, always containing steps-1 and 0;
  * ``ddpm_coef``             -- ancestral sampling (sigma^2 = beta', the reference's choice) over a sub-sequence;
                                 over *all* timesteps it reproduces the reference's table;
  * ``ddim_coef``             -- DDIM with stochasticity eta (eta = 0: deterministic);
  * ``shifted_cosine_betas``  -- the cosine schedule with its SNR multiplied by scale^2 (logSNR shift 2 log scale);
  * ``dpmpp_2m_coef``         -- DPM-Solver++(2M) (Lu et al. 2022, "DPM-Solver++", Alg. 2) and its SDE variant: a second-order
                                 multistep update that also carries the previous step's x0 prediction (a [diffusion_steps, 6]
                                 table for ``ditto_engine_load_multistep_table``);
  * ``known_coef``            -- known frames (speech prompt, infilling): the re-noising rows {sqrt(abar_next),
                                 sqrt(1 - abar_next)} of replacement conditioning (a [diffusion_steps, 2] table for
                                 ``ditto_engine_load_known_table``).
"""
from __future__ import annotations

from typing import Sequence

import torch

__all__ = ["spaced_timesteps", "ddpm_coef", "ddim_coef", "dpmpp_2m_coef", "known_coef", "shifted_cosine_betas", "coef_table"]


def spaced_timesteps(train_steps: int, num_steps: int) -> torch.Tensor:
    """``num_steps`` model timesteps out of ``range(train_steps)``, descending, first = train_steps-1, last = 0."""
    if not 1 <= num_steps <= train_steps:
        raise ValueError("need 1 <= num_steps <= diffusion_steps")
    if num_steps == 1:
        return torch.tensor([train_steps - 1], dtype=torch.int64)
    d = num_steps - 1     # evenly spaced, rounded half up, in integer arithmetic (no float ties)
    i = torch.arange(num_steps, dtype=torch.int64)
    tau = (2 * (train_steps - 1) * (d - i) + d) // (2 * d)
    if torch.unique(tau).numel() != num_steps:
        raise ValueError("spaced_timesteps: duplicate timesteps")
    return tau


def _acp_pairs(alphas_cumprod: torch.Tensor, taus: Sequence[int]):
    acp = alphas_cumprod.to(torch.float64)
    taus = [int(t) for t in taus]
    if any(a <= b for a, b in zip(taus, taus[1:])) or taus[-1] < 0 or taus[0] >= acp.numel():
        raise ValueError("timesteps must be strictly descending and inside the schedule")
    a_t = acp[taus]
    a_p = torch.cat([acp[taus[1:]], torch.ones(1, dtype=torch.float64)])   # "previous" of the last visited step: abar = 1
    return taus, a_t, a_p


def ddpm_coef(alphas_cumprod: torch.Tensor, taus: Sequence[int]) -> torch.Tensor:
    """Ancestral sampling over the visited timesteps: alpha' = abar_t / abar_prev, sigma^2 = beta' = 1 - alpha' (the
    reference's variance choice, SpeechGenerator.py:143-145), no noise on the last visited step (its ``t > 0`` mask).
    Returns float64 [len(taus), 3]."""
    taus, a_t, a_p = _acp_pairs(alphas_cumprod, taus)
    al = a_t / a_p
    c1 = 1.0 / al.sqrt()
    c2 = (1.0 - al) / (1.0 - a_t).sqrt()
    c3 = (1.0 - al).sqrt()
    c3[-1] = 0.0
    return torch.stack([c1, c2, c3], dim=1)


def ddim_coef(alphas_cumprod: torch.Tensor, taus: Sequence[int], eta: float = 0.0) -> torch.Tensor:
    """DDIM: x0 = (x - sqrt(1-abar_t) eps)/sqrt(abar_t); x_prev = sqrt(abar_p) x0 + sqrt(1-abar_p-sigma^2) eps + sigma z,
    sigma = eta sqrt((1-abar_p)/(1-abar_t)) sqrt(1-abar_t/abar_p), rewritten as c1 (x - c2 eps) + c3 z."""
    taus, a_t, a_p = _acp_pairs(alphas_cumprod, taus)
    sigma = float(eta) * ((1.0 - a_p) / (1.0 - a_t)).sqrt() * (1.0 - a_t / a_p).clamp_min(0.0).sqrt()
    c1 = (a_p / a_t).sqrt()
    c2 = (1.0 - a_t).sqrt() - (1.0 - a_p - sigma * sigma).clamp_min(0.0).sqrt() / c1
    return torch.stack([c1, c2, sigma], dim=1)


def dpmpp_2m_coef(alphas_cumprod: torch.Tensor, taus: Sequence[int], eta: float = 0.0) -> torch.Tensor:
    """DPM-Solver++(2M) over the visited timesteps tau_0 > ... > tau_{K-1}, with stochasticity eta in [0, 1] (0: the ODE
    solver of Lu et al. 2022, Alg. 2; 1: the "midpoint" 2M-SDE, rewritten for the VP process).  With
    alpha_i = sqrt(abar_{tau_i}), sigma_i = sqrt(1 - abar_{tau_i}), abar_K = 1, lambda_i = log(alpha_i / sigma_i),
    h_i = lambda_{i+1} - lambda_i, the step is

        x0_i    = (x_i - sigma_i eps_i) / alpha_i
        D_i     = x0_i                                        i == 0 or i == K-1 (first order)
                = x0_i + (x0_i - x0_{i-1}) / (2 r_i),         r_i = h_{i-1} / h_i, otherwise
        x_{i+1} = (sigma_{i+1}/sigma_i) e^{-eta h_i} x_i + alpha_{i+1} (1 - e^{-(1+eta) h_i}) D_i
                  + sigma_{i+1} sqrt(1 - e^{-2 eta h_i}) z

    and the last one returns x0_{K-1} without noise.  Rewritten for the device kernel as

        x_out = c1 (x - c2 eps) + c3 z + c4 hist,     hist <- d1 (x - d2 eps)   (= x0_i, read by the next step)

    with k = 1/(2 r_i) (0 on first-order steps), phi = alpha_{i+1} (1 - e^{-(1+eta) h}), rho = (sigma_{i+1}/sigma_i) e^{-eta h}:
    c1 = rho + phi (1+k) / alpha_i, c2 = phi (1+k) sigma_i / (alpha_i c1), c3 = sigma_{i+1} sqrt(1 - e^{-2 eta h}),
    c4 = -phi k, d1 = 1/alpha_i, d2 = sigma_i.  The first and last rows have c4 = 0; the last row equals DDIM's.  A
    first-order step equals ``ddim_coef`` at eta = 0 and eta = 1; for 0 < eta < 1 the two families inject noise
    differently (DDIM's eta scales its sigma_t, this one the exponent) and are different samplers.
    Returns float64 [len(taus), 6]."""
    eta = float(eta)
    if not 0.0 <= eta <= 1.0:
        raise ValueError("dpmpp_2m_coef: eta must be in [0, 1]")
    taus, a_t, a_p = _acp_pairs(alphas_cumprod, taus)
    al, sg = a_t.sqrt(), (1.0 - a_t).sqrt()
    out = torch.zeros((len(taus), 6), dtype=torch.float64)
    out[:, 4], out[:, 5] = 1.0 / al, sg
    out[-1, 0], out[-1, 1] = (a_p[-1] / a_t[-1]).sqrt(), sg[-1]      # x_K = x0_{K-1}: DDIM's last row
    if len(taus) > 1:
        a, s, a1, s1 = al[:-1], sg[:-1], a_p[:-1].sqrt(), (1.0 - a_p[:-1]).sqrt()
        lam = (al / sg).log()
        h = lam[1:] - lam[:-1]                                           # h_i, i < K-1
        k = torch.zeros_like(h)
        k[1:] = h[1:] / (2.0 * h[:-1])                                   # 1 / (2 r_i) on the second-order steps
        phi = a1 * -torch.expm1(-(1.0 + eta) * h)
        rho = s1 / s * torch.exp(-eta * h)
        c1 = rho + phi * (1.0 + k) / a
        out[:-1, 0] = c1
        out[:-1, 1] = phi * (1.0 + k) * s / (a * c1)
        out[:-1, 2] = s1 * (-torch.expm1(-2.0 * eta * h)).sqrt()
        out[:-1, 3] = -phi * k
    return out


def known_coef(alphas_cumprod: torch.Tensor, taus: Sequence[int]) -> torch.Tensor:
    """Replacement conditioning (Song et al. 2021, score SDE, "imputation"): the step that starts at tau_i writes a known
    frame as q(x_{i+1} | p) = sqrt(abar_next) p + sqrt(1 - abar_next) z, abar_next = abar_{tau_{i+1}} of THIS schedule (the
    sampler's own cumprod, not the model's betas buffer) and 1 after the last visited step, whose row {1, 0} returns p.
    Returns float64 [len(taus), 2] = {sqrt(abar_next), sqrt(1 - abar_next)}."""
    _, _, a_p = _acp_pairs(alphas_cumprod, taus)
    return torch.stack([a_p.sqrt(), (1.0 - a_p).sqrt()], dim=1)


def shifted_cosine_betas(timesteps: int, scale: float, s: float = 0.008) -> torch.Tensor:
    """DiTTO.cosine_beta_schedule (DiTTO.py:96-104) with the signal-to-noise ratio of every level multiplied by scale^2
    (abar' = scale^2 abar / (scale^2 abar + 1 - abar)); scale = 1 returns the reference's betas (same clip)."""
    x = torch.linspace(0, timesteps, timesteps + 1, dtype=torch.float64)
    acp = torch.cos(((x / timesteps) + s) / (1 + s) * torch.pi * 0.5) ** 2
    acp = acp / acp[0]
    k = float(scale) ** 2
    acp = k * acp / (k * acp + 1.0 - acp)
    betas = 1.0 - acp[1:] / acp[:-1]
    return torch.clip(betas, 0.0001, 0.9999).to(torch.float32)


def coef_table(diffusion_steps: int, taus: Sequence[int], coef: torch.Tensor) -> torch.Tensor:
    """Scatter per-visited-step rows into the engine's [diffusion_steps, 3] fp32 table, its [diffusion_steps, 6] multistep
    table for 6-column rows or its [diffusion_steps, 2] known-frame table for 2-column rows (unvisited rows: identity,
    c1 = d1 = 1; {1, 0} for known frames)."""
    if coef.dim() != 2 or coef.shape[1] not in (2, 3, 6):
        raise ValueError("coef_table: rows must have 2, 3 or 6 columns")
    tab = torch.zeros((diffusion_steps, coef.shape[1]), dtype=torch.float32)
    tab[:, 0] = 1.0
    if coef.shape[1] == 6:
        tab[:, 4] = 1.0
    tab[torch.as_tensor([int(t) for t in taus])] = coef.to(torch.float32)
    return tab
