"""CPU checks of sampling around known frames (speech prompt, infilling): the known-frame table (schedules.known_coef) against
the sampler's own schedule, the properties of the textbook replacement sampler of oracle/known_ref.py, and the C-ABI surface
of the known-frame entry points."""
import ctypes
import os
import re

import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib, build, schedules as S
from oracle import ditto_oracle as O
from oracle import known_ref as KR
from oracle import multistep_ref as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cpu_sampler(monkeypatch, steps, **kw):
    """A DiTTOSampler on a CPU model: its host tables only (the engine is never touched)."""
    monkeypatch.setattr(D.DiTTOSampler, "_activate", lambda self, known=False: None)
    m = D.DiTTO(hidden_dim=64, num_layers=1, num_heads=2, time_dim=32, text_dim=64, diffusion_steps=steps)
    return m, D.DiTTOSampler(m, 3.0, **kw)


SAMPLERS = [("ddpm-all", {})] + [(f"{m}-{k}", dict(method=m, num_steps=k)) for m in ("ddim", "dpmpp_2m") for k in (2, 5, 16, 50)]


@pytest.mark.parametrize("steps,scale", [(50, None), (1000, None), (50, 0.3)])
@pytest.mark.parametrize("name,kw", SAMPLERS, ids=[n for n, _ in SAMPLERS])
def test_known_table_is_the_samplers_own_schedule(monkeypatch, steps, scale, name, kw):
    m, s = cpu_sampler(monkeypatch, steps, schedule_scale=scale, **kw)
    betas = O.cosine_beta_schedule(steps) if scale is None else O.shifted_cosine_betas(steps, scale)
    acp = torch.cumprod(1.0 - betas.double(), dim=0)
    taus = s.timesteps.tolist()
    assert taus == O.spaced_timesteps(steps, kw.get("num_steps", steps))
    coef = S.known_coef(acp, taus)
    assert coef.dtype == torch.float64 and coef.shape == (len(taus), 2)
    for i in range(len(taus)):
        a_next = float(acp[taus[i + 1]]) if i + 1 < len(taus) else 1.0
        assert coef[i, 0].item() == pytest.approx(a_next ** 0.5, rel=1e-15, abs=0.0)
        assert coef[i, 1].item() == pytest.approx((1.0 - a_next) ** 0.5, rel=1e-15, abs=1e-300)
    assert coef[-1].tolist() == [1.0, 0.0]
    # the sampler's [steps, 2] table: its rows at the visited timesteps, {1, 0} elsewhere
    tab = s.known_table
    assert tab.shape == (steps, 2) and tab.dtype == torch.float32
    assert torch.equal(tab[taus], coef.float())
    unvisited = sorted(set(range(steps)) - set(taus))
    assert torch.equal(tab[unvisited], torch.tensor([1.0, 0.0]).expand(len(unvisited), 2))
    # not the model's "alphas_cumprod" buffer: it holds the reference schedule's betas (DiTTO.py:63-64)
    buf = m.alphas_cumprod.double()
    wrong = torch.stack([buf[taus[1:]].sqrt(), (1.0 - buf[taus[1:]]).sqrt()], dim=1)
    assert not torch.allclose(coef[:-1], wrong, rtol=1e-3, atol=1e-3)


def test_coef_table_takes_two_columns():
    acp = torch.cumprod(1.0 - O.cosine_beta_schedule(50).double(), dim=0)
    taus = S.spaced_timesteps(50, 10).tolist()
    tab = S.coef_table(50, taus, S.known_coef(acp, taus))
    assert tab.shape == (50, 2)
    with pytest.raises(ValueError, match="2, 3 or 6"):
        S.coef_table(50, taus, torch.zeros(10, 4, dtype=torch.float64))


# ------------------------------------------------------------------------------------------------ oracle properties
@pytest.fixture(scope="module")
def small():
    cfg = O.OracleConfig(32, 1, 2, 16, 32, 12)
    sd = O.make_state_dict(cfg, 3)
    x, text, noise = O.make_inputs(2, 10, 4, cfg, 4, steps_noise=12)
    known = torch.randn(2, 10, 32, generator=torch.Generator().manual_seed(9))
    return cfg, sd, x, text, noise, known


RUNS = [dict(method="ddpm"), dict(method="ddim", num_steps=5, eta=0.5), dict(method="ddpm", num_steps=4, schedule_scale=0.3),
        dict(method="dpmpp_2m", num_steps=6), dict(method="dpmpp_2m", num_steps=6, eta=1.0)]


def _plain(small, w, kw):
    cfg, sd, x, text, noise, _ = small
    if kw["method"] == "dpmpp_2m":
        return M.sample_latents_dpmpp_2m(sd, cfg, text, x, noise, w, **{k: v for k, v in kw.items() if k != "method"})
    return O.sample_latents_variant(sd, cfg, text, x, noise, w, **kw)


@pytest.mark.parametrize("kw", RUNS, ids=lambda k: "-".join(f"{a}={b}" for a, b in k.items()))
@pytest.mark.parametrize("w", [3.0, None], ids=["w3", "unguided"])
def test_oracle_all_false_mask_is_the_plain_sampler(small, kw, w):
    cfg, sd, x, text, noise, known = small
    got = KR.sample_latents_known(sd, cfg, text, x, noise, known, torch.zeros(2, 10, dtype=torch.bool), w, **kw)
    assert torch.equal(got, _plain(small, w, kw))


@pytest.mark.parametrize("kw", RUNS, ids=lambda k: "-".join(f"{a}={b}" for a, b in k.items()))
def test_oracle_keeps_known_frames(small, kw):
    cfg, sd, x, text, noise, known = small
    mask = torch.zeros(2, 10, dtype=torch.bool)
    mask[0, :4] = True                   # a prompt to continue
    mask[1] = True
    mask[1, 3:7] = False                 # a span to fill
    got = KR.sample_latents_known(sd, cfg, text, x, noise, known, mask, 3.0, **kw)
    assert torch.equal(got[mask], known[mask])
    free = _plain(small, 3.0, kw)
    assert not torch.allclose(got[~mask], free[~mask])        # the known frames steer the others
    every = KR.sample_latents_known(sd, cfg, text, x, noise, known, torch.ones(2, 10, dtype=torch.bool), 3.0, **kw)
    assert torch.equal(every, known)


# ------------------------------------------------------------------------------------------------ C-ABI surface
KNOWN_ABI = ["ditto_engine_load_known_table", "ditto_cfg_update_known", "ditto_p_sample_known", "ditto_p_sample_ragged_known"]


def test_known_abi_declared_bound_and_exported():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "ditto_b200.h")).read(), flags=re.S)
    lib = ctypes.CDLL(build.build())
    for name in KNOWN_ABI:
        m = re.search(r"\b" + name + r"\s*\(([^)]*)\)", src)
        assert m, f"{name} not declared in include/ditto_b200.h"
        n_args = len([a for a in m.group(1).split(",") if a.strip()])
        assert len(_lib.SIGNATURES[name][1]) == n_args, name
        assert hasattr(lib, name), name
    assert lib.ditto_abi_version() == 1
