"""Full-size parity (-m gpu) against outputs of the UNMODIFIED reference (tests/golden/full_traj.npz, minted by
tests/golden/make_golden_full.py) at the shapes BASELINE.json names, repo-default model (H = 768, L = 5, one head of 768):
  * C1/C2 utterance: the full 50-step CFG sampling loop at T = 750, S = 64 -- first / last guided eps_hat and final latent;
  * C3 utterance: one forward at T = 2250, S = 192, all five layers;
  * C5: three speech-length-predictor-sized utterances (2 s / 11 s / 20 s) sampled TOGETHER through the packed ragged path,
    each against its own per-utterance (unpadded) reference run;
  * C4 size (128 utterances on one GPU, M = 192 000 rows): batch independence against the same utterances run in a batch of 2.
Bars (BASELINE.json): rel-L2 <= 1e-4 fp32 path, <= 2e-2 bf16 path."""
import numpy as np
import pytest
import torch

import ditto_tts_b200 as D
from oracle import ditto_oracle as O  # checker only (weights / inputs regenerate from seeds)

pytestmark = pytest.mark.gpu
BAR = {"fp32": 1e-4, "bf16": 2e-2}


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def traj(golden):
    return golden("full_traj.npz")


def rel(a, b):
    return O.rel_l2(a.float().cpu(), b.float().cpu())


def model_for(traj, precision, dev):
    H, L, heads, Td, Xd, steps, wseed, stride = (int(v) for v in traj["meta"])
    cfg = O.OracleConfig(H, L, heads, Td, Xd, steps)
    m = D.DiTTO(hidden_dim=H, num_layers=L, num_heads=heads, time_dim=Td, text_dim=Xd, diffusion_steps=steps, precision=precision)
    m.load_state_dict(O.make_state_dict(cfg, wseed), strict=True)
    return m.to(dev), cfg, stride


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_c1_50_step_cfg_trajectory_full_size(dev, traj, precision):
    m, cfg, stride = model_for(traj, precision, dev)
    seed, T, S = (int(v) for v in traj["c1_traj::shape"])
    x, text, noise = O.make_inputs(1, T, S, cfg, seed=seed, steps_noise=cfg.diffusion_steps)
    s = D.DiTTOSampler(m, guidance_scale=float(traj["w"][0]))
    rec = []
    out = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise.to(dev), record=rec)
    assert rel(rec[0][:, ::stride], torch.from_numpy(traj["c1_traj::eps_first_sub"])) <= BAR[precision]
    assert rel(rec[-1][:, ::stride], torch.from_numpy(traj["c1_traj::eps_last_sub"])) <= BAR[precision]
    assert rel(out[:, ::stride], torch.from_numpy(traj["c1_traj::final_sub"])) <= BAR[precision]
    norms = np.array([float(e.double().norm()) for e in rec])
    assert np.allclose(norms, traj["c1_traj::eps_norms"], rtol=BAR[precision])
    assert abs(float(out.double().norm()) / traj["c1_traj::norms"][2] - 1.0) <= BAR[precision]
    # the product's own stepping (CUDA-graph replay) on the same supplied noise
    graph_out = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise.to(dev))
    assert rel(graph_out, out) <= 1e-6


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_c3_forward_30s_all_layers(dev, traj, precision):
    m, cfg, stride = model_for(traj, precision, dev)
    seed, T, S, t_val = (int(v) for v in traj["c3_fwd::shape"])
    x, text, _ = O.make_inputs(1, T, S, cfg, seed=seed)
    out = m(x.to(dev), text.to(dev), torch.tensor([t_val]).to(dev))
    assert rel(out[:, ::stride], torch.from_numpy(traj["c3_fwd::out_sub"])) <= BAR[precision]
    assert abs(float(out.double().norm()) / traj["c3_fwd::norms"][0] - 1.0) <= BAR[precision]
    if precision == "bf16":   # the C3 batch shape (4 x 30 s): every utterance of the batch equals the single-utterance run
        xb = torch.cat([x, x.flip(1), x * 0.5, x]).to(dev)
        tb = torch.cat([text, text.flip(1), text, text * 2]).to(dev)
        ob = m(xb, tb, torch.tensor([t_val, 3, 49, t_val]).to(dev))
        assert rel(ob[0:1], out) <= 1e-5


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_c5_three_utterances_sampled_together_vs_per_utterance_reference(dev, traj, precision):
    m, cfg, stride = model_for(traj, precision, dev)
    names = ["c5_u0", "c5_u1", "c5_u2"]
    xs, texts, noises, lengths = [], [], [], []
    for n in names:
        seed, T, S = (int(v) for v in traj[f"{n}::shape"])
        x, text, noise = O.make_inputs(1, T, S, cfg, seed=seed, steps_noise=cfg.diffusion_steps)
        xs.append(x[0].to(dev)); texts.append(text[0].to(dev)); noises.append(noise[:, 0].to(dev)); lengths.append(T)
    s = D.DiTTOSampler(m, guidance_scale=float(traj["w"][0]))
    rec = []
    outs = s.sample_latents_ragged(texts, lengths, x_init=xs, noise=noises, record=rec)
    for i, n in enumerate(names):
        assert rel(rec[0][i][::stride], torch.from_numpy(traj[f"{n}::eps_first_sub"])[0]) <= BAR[precision], n
        assert rel(rec[-1][i][::stride], torch.from_numpy(traj[f"{n}::eps_last_sub"])[0]) <= BAR[precision], n
        e = rel(outs[i][::stride], torch.from_numpy(traj[f"{n}::final_sub"])[0])
        assert e <= BAR[precision], (n, e)
        # norms of the full tensors: every frame, not only the stored ones
        assert abs(float(outs[i].double().norm()) / traj[f"{n}::norms"][2] - 1.0) <= BAR[precision], n
        norms = np.array([float(r[i].double().norm()) for r in rec])
        assert np.allclose(norms, traj[f"{n}::eps_norms"], rtol=BAR[precision]), n
    graph_outs = s.sample_latents_ragged(texts, lengths, x_init=xs, noise=noises)      # CUDA-graph stepping, same noise
    for a, b in zip(graph_outs, outs):
        assert rel(a, b) <= 1e-6


def test_c4_size_batch_independence(dev):
    """BASELINE C4 on fewer GPUs: 128 utterances x 10 s on one GPU (2 x 128 sequences, M = 192 000 rows, 5.6 GB workspace).
    One guided sampler step; utterances of the big batch equal the same utterances run in a batch of two."""
    cfg = O.OracleConfig(768, 5, 1, 256, 768, 50)
    m = D.DiTTO(hidden_dim=768, num_layers=5, num_heads=1, time_dim=256, text_dim=768, diffusion_steps=50, precision="bf16")
    m.load_state_dict(O.make_state_dict(cfg, 0), strict=True)
    m = m.to(dev)
    s = D.DiTTOSampler(m)
    B, T, S = 128, 750, 64
    g = torch.Generator(device=dev).manual_seed(77)
    x = torch.randn(B, T, 768, device=dev, generator=g)
    text = torch.randn(B, S, 768, device=dev, generator=g)
    z = torch.randn(B, T, 768, device=dev, generator=g)
    t = torch.full((B,), 31, dtype=torch.long, device=dev)
    full = s.p_sample(x, t, text, noise=z, guidance_scale=3.0)
    assert bool(torch.isfinite(full).all())
    for i in (0, 77, 127):
        j = (i + 5) % B
        idx = torch.tensor([i, j], device=dev)
        pair = s.p_sample(x[idx], t[:2], text[idx], noise=z[idx], guidance_scale=3.0)
        assert rel(full[idx], pair) <= 1e-5, i
    del full
    torch.cuda.empty_cache()
