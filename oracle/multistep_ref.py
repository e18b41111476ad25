"""DPM-Solver++(2M) written the textbook way  --  TEST INFRASTRUCTURE ONLY.

An EXTENSION like the sampler variants of ditto_oracle.py (the reference has one sampler): the multistep solver of Lu et al.
2022, "DPM-Solver++", Alg. 2 (eta = 0), and its SDE variant (eta = 1: the "midpoint" 2M-SDE, rewritten for the VP
process), stated in lambda = log(alpha / sigma), step by step, in float64.  It does NOT use the c1..c4 / d1, d2 rewrite
the product's kernel reads (ditto_tts_b200/schedules.py: dpmpp_2m_coef), so the two can be checked against each other.

Visited timesteps tau_0 > ... > tau_{K-1} = 0 (ditto_oracle.spaced_timesteps), alpha_i = sqrt(abar_{tau_i}),
sigma_i = sqrt(1 - abar_{tau_i}), h_i = lambda_{i+1} - lambda_i:

    x0_i    = (x_i - sigma_i eps_i) / alpha_i
    D_i     = x0_i                                      on the first step
            = x0_i + (x0_i - x0_{i-1}) / (2 r_i),       r_i = h_{i-1} / h_i, otherwise
    x_{i+1} = (sigma_{i+1}/sigma_i) e^{-eta h_i} x_i + alpha_{i+1} (1 - e^{-(1+eta) h_i}) D_i + sigma_{i+1} sqrt(1 - e^{-2 eta h_i}) z

and the last step (abar_K = 1, h = inf) returns x0_{K-1}.
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import torch

from . import ditto_oracle as O

Tensor = torch.Tensor


def log_snr(acp: float) -> float:
    """lambda = log(alpha / sigma) of one noise level abar."""
    return 0.5 * math.log(acp / (1.0 - acp))


def dpmpp_2m_update(x: Tensor, eps: Tensor, z: Tensor, acp_t: float, acp_next: Optional[float], eta: float,
                    x0_prev: Optional[Tensor] = None, h_prev: Optional[float] = None) -> Tuple[Tensor, Tensor, Optional[float]]:
    """One step from abar_t to abar_next (None: the last step, to the data) in float64.
    -> (x_next cast to x.dtype, x0 of this step in float64, h of this step: the history of the next one)."""
    xd, ed = x.double(), eps.double()
    a, s = math.sqrt(acp_t), math.sqrt(1.0 - acp_t)
    x0 = (xd - s * ed) / a
    if acp_next is None:
        return x0.to(x.dtype), x0, None
    a1, s1 = math.sqrt(acp_next), math.sqrt(1.0 - acp_next)
    h = log_snr(acp_next) - log_snr(acp_t)
    if x0_prev is None:
        d = x0
    else:
        r = h_prev / h
        d = x0 + (x0 - x0_prev) / (2.0 * r)
    out = (s1 / s) * math.exp(-eta * h) * xd + a1 * (-math.expm1(-(1.0 + eta) * h)) * d
    if eta > 0.0:
        out = out + s1 * math.sqrt(-math.expm1(-2.0 * eta * h)) * z.double()
    return out.to(x.dtype), x0, h


def sample_latents_dpmpp_2m(sd, cfg: O.OracleConfig, text_emb: Tensor, x_init: Tensor, noise: Tensor,
                            guidance_scale: Optional[float] = None, num_steps: Optional[int] = None, eta: float = 0.0,
                            schedule_scale: Optional[float] = None, record: Optional[List[Tensor]] = None) -> Tensor:
    """ditto_oracle.sample_latents_variant with the 2M update: same arguments (noise index = t_val), same schedules."""
    steps = cfg.diffusion_steps
    betas = O.cosine_beta_schedule(steps) if schedule_scale is None else O.shifted_cosine_betas(steps, schedule_scale)
    acp = torch.cumprod(1.0 - betas.double(), dim=0).tolist()
    taus = O.spaced_timesteps(steps, steps if num_steps is None else num_steps)
    x, x0_prev, h_prev = x_init, None, None
    for i, t_val in enumerate(taus):
        t = torch.full((x.shape[0],), t_val, dtype=torch.long)
        eps = O.predict_noise(sd, cfg, x, text_emb, t, guidance_scale)
        if record is not None:
            record.append(eps)
        acp_next = acp[taus[i + 1]] if i + 1 < len(taus) else None
        x, x0_prev, h_prev = dpmpp_2m_update(x, eps, noise[t_val], acp[t_val], acp_next, eta, x0_prev, h_prev)
    return x
