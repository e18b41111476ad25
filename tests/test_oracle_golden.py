"""Pin the CPU oracle (oracle/ditto_oracle.py) to outputs of the unmodified reference.

The fixtures under tests/golden/ were produced by tests/golden/make_golden.py, which imports the
reference modules from /root/reference/src (DiTTO.py, DiT.py, SpeechGenerator.__p_sample).
Bars: fp32 restatement vs reference fp32: rel-L2 <= 2e-6 (re-association noise; the reference's own
fp32-vs-fp64 noise floor is 4e-7, SURVEY.md 8c).  Schedules: bit-exact.
"""
import numpy as np
import pytest
import torch

from oracle import ditto_oracle as O

FP32_BAR = 2e-6


def _cfg(a):
    return O.OracleConfig(*[int(v) for v in a[:6]])


def test_schedule_bit_exact(golden):
    g = golden("schedules.npz")
    for steps in (50, 1000):
        betas, alphas, ac = O.sampler_tables(steps)
        assert np.array_equal(betas.numpy(), g[f"betas{steps}"])
        assert np.array_equal(ac.numpy(), g[f"alphas_cumprod{steps}"])
    # known answers quoted in SURVEY.md section 8 a11
    b50, _, ac50 = O.sampler_tables(50)
    assert abs(float(b50[0]) - 1.747e-3) < 1e-6 and float(b50[49]) == pytest.approx(0.9999)
    assert float(ac50[49]) == pytest.approx(9.71e-8, rel=1e-2)
    b1000, _, ac1000 = O.sampler_tables(1000)
    assert float(b1000[0]) == pytest.approx(1e-4) and float(ac1000[999]) == pytest.approx(2.43e-10, rel=1e-2)


def test_tiny_forward_and_taps(golden):
    g = golden("tiny_full.npz")
    cfg = _cfg(g["cfg"])
    sd = {k[4:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd::")}
    x, text, t = (torch.from_numpy(g[k]) for k in ("x", "text", "t"))
    taps = {}
    out = O.ditto_forward(sd, cfg, x, text, t, taps)
    assert O.rel_l2(out, torch.from_numpy(g["out"])) <= FP32_BAR
    for k in ("adaln", "block0", "block1"):
        assert O.rel_l2(taps[k], torch.from_numpy(g["tap::" + k])) <= FP32_BAR, k
    assert np.allclose(O.rotary_angles(x.shape[1], cfg.head_dim).numpy(), g["rotary"], rtol=0, atol=0)


def test_tiny_weights_regenerate(golden):
    """make_state_dict is deterministic across boxes: the stored weights equal a fresh draw."""
    g = golden("tiny_full.npz")
    cfg = _cfg(g["cfg"])
    sd = O.make_state_dict(cfg, seed=3)
    for k in g.files:
        if k.startswith("sd::"):
            assert np.array_equal(sd[k[4:]].numpy(), g[k]), k
    x, text, noise = O.make_inputs(2, 24, 8, cfg, seed=4, steps_noise=cfg.diffusion_steps)
    assert np.array_equal(x.numpy(), g["x"]) and np.array_equal(text.numpy(), g["text"])


def test_tiny_reference_sampler_loop(golden):
    """The reference's own __p_sample loop (no guidance), noise replayed from its seeded randn_like."""
    g = golden("tiny_full.npz")
    cfg = _cfg(g["cfg"])
    sd = {k[4:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd::")}
    x, text = torch.from_numpy(g["x"]), torch.from_numpy(g["text"])
    noise = torch.from_numpy(g["ref_noise"])
    rec = []
    out = O.sample_latents(sd, cfg, text, x, noise, guidance_scale=None, record=rec)
    assert len(rec) == cfg.diffusion_steps
    assert O.rel_l2(out, torch.from_numpy(g["sampled"])) <= 1e-5
    qs = O.q_sample(sd, x, torch.from_numpy(g["t"]), torch.from_numpy(g["q_noise"]))
    assert O.rel_l2(qs, torch.from_numpy(g["q_sample"])) <= 1e-7


@pytest.mark.parametrize("name", ["c1_default", "ctor_default", "ragged"])
def test_full_size_forward(golden, name):
    g = golden("full_size.npz")
    meta = [int(v) for v in g[f"{name}::meta"]]
    cfg = O.OracleConfig(*meta[:6])
    wseed, iseed, B, T, S, stride = meta[6:]
    sd = O.make_state_dict(cfg, seed=wseed)
    x, text, _ = O.make_inputs(B, T, S, cfg, seed=iseed)
    t = torch.from_numpy(g[f"{name}::t"])
    taps = {}
    out = O.ditto_forward(sd, cfg, x, text, t, taps)
    assert O.rel_l2(out[:, ::stride], torch.from_numpy(g[f"{name}::out_sub"])) <= FP32_BAR
    assert float(out.double().norm()) == pytest.approx(float(g[f"{name}::out_norm"][0]), rel=1e-5)
    assert O.rel_l2(taps["adaln"][:, ::stride], torch.from_numpy(g[f"{name}::adaln_sub"])) <= FP32_BAR
    assert O.rel_l2(taps["block0"][:, ::stride], torch.from_numpy(g[f"{name}::block0_sub"])) <= FP32_BAR


def test_cfg_trajectory_endpoints(golden):
    """50-step CFG (w=3, uncond = zero text) on the default model: first/last eps_hat and final latent
    of the reference-forward trajectory (every `stride`-th frame, plus the norms of the full tensors).
    The oracle runs the same loop (2 forwards per step)."""
    g = golden("cfg_traj.npz")
    B, T, S, iseed, wseed, steps = [int(v) for v in g["meta"]]
    stride = int(g["stride"][0])
    cfg = O.OracleConfig(768, 5, 1, 256, 768, steps)
    sd = O.make_state_dict(cfg, seed=wseed)
    x, text, noise = O.make_inputs(B, T, S, cfg, seed=iseed, steps_noise=steps)
    rec = []
    final = O.sample_latents(sd, cfg, text, x, noise, guidance_scale=float(g["w"][0]), record=rec)
    assert O.rel_l2(rec[0][:, ::stride], torch.from_numpy(g["eps_first"])) <= FP32_BAR
    # chaotic growth of the latent (rms ~1e5 after 50 steps) amplifies fp32 re-association noise
    assert O.rel_l2(rec[-1][:, ::stride], torch.from_numpy(g["eps_last"])) <= 1e-4
    assert O.rel_l2(final[:, ::stride], torch.from_numpy(g["final"])) <= 1e-4
    assert float(final.double().norm()) == pytest.approx(float(g["final_norm"][0]), rel=1e-4)
    norms = np.array([float(e.double().norm()) for e in rec])
    assert np.allclose(norms, g["eps_norms"], rtol=1e-4)
