"""CPU checks of the DPM-Solver++(2M) sampler (schedules.dpmpp_2m_coef): its c-form table against the textbook lambda-form
of oracle/multistep_ref.py step by step, its pins to DDIM, its order of convergence on toys with exact denoisers, and
the C-ABI surface of the multistep entry points."""
import ctypes
import math
import os
import re

import pytest
import torch

from ditto_tts_b200 import _lib, build, schedules as S
from oracle import ditto_oracle as O
from oracle import multistep_ref as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def acp64(steps, scale=None):
    betas = O.cosine_beta_schedule(steps) if scale is None else O.shifted_cosine_betas(steps, scale)
    return torch.cumprod(1.0 - betas.double(), dim=0)


def c_form_step(row, x, eps, z, hist):
    """The kernel's arithmetic in float64: x_out = c1 (x - c2 eps) + c3 z + c4 hist (hist skipped when c4 == 0),
    hist <- d1 (x - d2 eps)."""
    c1, c2, c3, c4, d1, d2 = (float(v) for v in row)
    out = c1 * (x - c2 * eps) + c3 * z
    if c4 != 0.0:
        out = out + c4 * hist
    return out, d1 * (x - d2 * eps)


@pytest.mark.parametrize("steps,scale", [(50, None), (1000, None), (50, 0.3), (1000, 0.3)])
@pytest.mark.parametrize("K", [2, 5, 16, 25, 50])
@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
def test_c_form_equals_lambda_form_every_step(steps, scale, K, eta):
    acp = acp64(steps, scale)
    taus = S.spaced_timesteps(steps, K).tolist()
    assert taus == O.spaced_timesteps(steps, K)
    coef = S.dpmpp_2m_coef(acp, taus, eta)
    assert coef.dtype == torch.float64 and coef.shape == (K, 6)
    g = torch.Generator().manual_seed(K)
    x = torch.randn(64, generator=g, dtype=torch.float64)
    xa, hist = x.clone(), torch.full_like(x, float("nan"))    # the history buffer holds garbage before the first step
    x0_prev = h_prev = None
    acp_l = acp.tolist()
    for i, t in enumerate(taus):
        eps, z = torch.randn(64, generator=g, dtype=torch.float64), torch.randn(64, generator=g, dtype=torch.float64)
        acp_next = acp_l[taus[i + 1]] if i + 1 < K else None
        x, x0_prev, h_prev = M.dpmpp_2m_update(x, eps, z, acp_l[t], acp_next, eta, x0_prev, h_prev)
        xa, hist = c_form_step(coef[i], xa, eps, z, hist)
        assert torch.isfinite(xa).all()
        assert float((xa - x).abs().max() / x.abs().max()) <= 1e-12, (i, t)


@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("steps,K", [(50, 16), (50, 50), (1000, 25), (20, 1)])
def test_first_and_last_rows(steps, K, eta):
    acp = acp64(steps)
    taus = S.spaced_timesteps(steps, K).tolist()
    coef = S.dpmpp_2m_coef(acp, taus, eta)
    assert coef[0, 3] == 0.0 and coef[-1, 3] == 0.0
    if K > 2:
        assert (coef[1:-1, 3] != 0.0).all()
    assert torch.equal(coef[-1, :3], S.ddim_coef(acp, taus, eta)[-1])      # x_K = x0_{K-1}, no noise
    assert torch.equal(coef[:, 4], 1.0 / acp[taus].sqrt()) and torch.equal(coef[:, 5], (1.0 - acp[taus]).sqrt())


@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("steps,scale", [(50, None), (1000, None), (50, 0.3)])
def test_two_steps_equal_ddim(steps, scale, eta):
    """K = 2: both steps are first order, and a first-order 2M(eta) step is DDIM(eta) for eta in {0, 1}."""
    acp = acp64(steps, scale)
    taus = S.spaced_timesteps(steps, 2).tolist()
    c2m, cddim = S.dpmpp_2m_coef(acp, taus, eta), S.ddim_coef(acp, taus, eta)
    assert (c2m[:, 3] == 0).all()
    torch.testing.assert_close(c2m[:, :3], cddim, rtol=1e-13, atol=1e-15)


def test_eta_range_and_table_layout():
    acp = acp64(50)
    taus = S.spaced_timesteps(50, 10).tolist()
    with pytest.raises(ValueError):
        S.dpmpp_2m_coef(acp, taus, 1.5)
    coef = S.dpmpp_2m_coef(acp, taus, 0.0)
    tab = S.coef_table(50, taus, coef)
    assert tab.shape == (50, 6) and tab.dtype == torch.float32
    assert torch.equal(tab[taus], coef.float())
    unvisited = sorted(set(range(50)) - set(taus))
    assert torch.equal(tab[unvisited], torch.tensor([1.0, 0, 0, 0, 1.0, 0]).expand(len(unvisited), 6))
    assert S.coef_table(50, taus, S.ddim_coef(acp, taus)).shape == (50, 3)      # the DDPM-form table is unchanged


# ------------------------------------------------------------------------------------------------ convergence
def run_c_form(coef, acp, taus, xT, eps_fn):
    """Deterministic sampling with the product's rows (float64) up to the state at tau_{K-1} = 0 (before the final
    x0 step).  Rows with 3 columns are DDIM's."""
    x, hist = xT.clone(), torch.full_like(xT, float("nan"))
    for i, t in enumerate(taus[:-1]):
        a = float(acp[t])
        eps = eps_fn(x, math.sqrt(a), math.sqrt(1.0 - a))
        row = coef[i] if coef.shape[1] == 6 else torch.cat([coef[i], torch.tensor([0.0, 1.0, 0.0], dtype=torch.float64)])
        x, hist = c_form_step(row, x, eps, torch.zeros_like(x), hist)
    return x


def test_order_of_convergence_gaussian():
    """x0 ~ N(mu, s^2): exact eps and a closed-form probability-flow ODE solution.  Doubling the step count cuts the error
    ~4x for 2M (second order) and ~2x for DDIM (first order)."""
    steps, mu, s = 1000, 0.7, 0.5
    acp = acp64(steps)
    xT = torch.randn(4096, generator=torch.Generator().manual_seed(0), dtype=torch.float64)

    def eps_fn(x, a, sg):
        return sg * (x - a * mu) / (a * a * s * s + sg * sg)

    def err(method, K):
        taus = S.spaced_timesteps(steps, K).tolist()
        coef = S.dpmpp_2m_coef(acp, taus, 0.0) if method == "2m" else S.ddim_coef(acp, taus, 0.0)
        x = run_c_form(coef, acp, taus, xT, eps_fn)
        aT, sT = math.sqrt(acp[taus[0]]), math.sqrt(1 - acp[taus[0]])
        a0, s0 = math.sqrt(acp[0]), math.sqrt(1 - acp[0])
        exact = a0 * mu + math.sqrt(a0 * a0 * s * s + s0 * s0) * (xT - aT * mu) / math.sqrt(aT * aT * s * s + sT * sT)
        return float((x - exact).norm() / exact.norm())

    r2m = err("2m", 33) / err("2m", 65)
    rddim = err("ddim", 33) / err("ddim", 65)
    assert r2m >= 3.5, r2m
    assert rddim <= 2.2, rddim


def test_mixture_25_steps_beat_ddim_50():
    """A three-component 1-D Gaussian mixture with its exact denoiser on the 50-step schedule: 2M at 25 steps has less than
    half the error of DDIM at 50, against an RK45 solution of the data-prediction ODE dy/dlambda = e^lambda x0(sigma y)."""
    from scipy.integrate import solve_ivp
    mu = torch.tensor([-1.5, 0.3, 1.8], dtype=torch.float64)
    sd = torch.tensor([0.15, 0.3, 0.1], dtype=torch.float64)
    pi = torch.tensor([0.3, 0.5, 0.2], dtype=torch.float64)

    def x0_star(x, a, sg):
        v = a * a * sd * sd + sg * sg
        w = torch.softmax(torch.log(pi) - 0.5 * torch.log(v) - 0.5 * (x[:, None] - a * mu) ** 2 / v, dim=1)
        return (w * (mu + a * sd * sd * (x[:, None] - a * mu) / v)).sum(1)

    def eps_fn(x, a, sg):
        return (x - a * x0_star(x, a, sg)) / sg

    steps = 50
    acp = acp64(steps)
    xT = torch.randn(2048, generator=torch.Generator().manual_seed(0), dtype=torch.float64)

    def f(lam, y):
        a = 1.0 / math.sqrt(1.0 + math.exp(-2.0 * lam))
        sg = a * math.exp(-lam)
        return math.exp(lam) * x0_star(torch.from_numpy(sg * y), a, sg).numpy()

    sol = solve_ivp(f, (M.log_snr(float(acp[-1])), M.log_snr(float(acp[0]))), (xT / math.sqrt(1 - acp[-1])).numpy(),
                    method="RK45", rtol=1e-10, atol=1e-10)
    ref = torch.from_numpy(sol.y[:, -1]) * math.sqrt(1 - acp[0])

    def err(coef_fn, K):
        taus = S.spaced_timesteps(steps, K).tolist()
        x = run_c_form(coef_fn(acp, taus, 0.0), acp, taus, xT, eps_fn)
        return float((x - ref).norm() / ref.norm())

    e2m, eddim = err(S.dpmpp_2m_coef, 25), err(S.ddim_coef, 50)
    assert e2m < 0.5 * eddim, (e2m, eddim)


# ------------------------------------------------------------------------------------------------ C-ABI surface
MULTISTEP_ABI = ["ditto_engine_load_multistep_table", "ditto_cfg_multistep_update", "ditto_cfg_multistep_update_rng",
                 "ditto_p_sample_multistep", "ditto_p_sample_multistep_rng", "ditto_p_sample_ragged_multistep",
                 "ditto_p_sample_ragged_multistep_rng"]


def test_multistep_abi_declared_bound_and_exported():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "ditto_b200.h")).read(), flags=re.S)
    lib = ctypes.CDLL(build.build())
    for name in MULTISTEP_ABI:
        m = re.search(r"\b" + name + r"\s*\(([^)]*)\)", src)
        assert m, f"{name} not declared in include/ditto_b200.h"
        n_args = len([a for a in m.group(1).split(",") if a.strip()])
        assert len(_lib.SIGNATURES[name][1]) == n_args, name
        assert hasattr(lib, name), name
    # each multistep entry point is its DDPM-form twin plus one pointer (hist)
    for ms, twin in [("ditto_cfg_multistep_update", "ditto_cfg_ddpm_update"),
                     ("ditto_cfg_multistep_update_rng", "ditto_cfg_ddpm_update_rng"),
                     ("ditto_p_sample_multistep", "ditto_p_sample"), ("ditto_p_sample_multistep_rng", "ditto_p_sample_rng"),
                     ("ditto_p_sample_ragged_multistep", "ditto_p_sample_ragged"),
                     ("ditto_p_sample_ragged_multistep_rng", "ditto_p_sample_ragged_rng")]:
        assert len(_lib.SIGNATURES[ms][1]) == len(_lib.SIGNATURES[twin][1]) + 1, ms
    assert lib.ditto_abi_version() == 1


def test_sampler_method_names():
    import ditto_tts_b200 as D
    m = D.DiTTO(hidden_dim=64, num_layers=1, num_heads=2, time_dim=32, text_dim=64, diffusion_steps=20)
    with pytest.raises(ValueError, match="dpmpp_2m"):
        D.DiTTOSampler(m, 3.0, method="dpmpp_3m")
