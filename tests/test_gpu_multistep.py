"""GPU checks of the DPM-Solver++(2M) sampler through the C-ABI (ditto_engine_load_multistep_table + ditto_p_sample_multistep
and friends): parity with the textbook lambda-form of oracle/multistep_ref.py, the kernel's pins to the DDPM-form update,
in-kernel noise, launch counts, table ownership between samplers, and the status codes of the entry points."""
import ctypes as C

import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib, schedules
from oracle import ditto_oracle as O
from oracle import multistep_ref as M

pytestmark = pytest.mark.gpu
BAR = {"fp32": 1e-4, "bf16": 2e-2}      # BASELINE.json: rel-L2 vs the fp32 oracle


def P(t):
    return C.c_void_p(t.data_ptr())


def ST():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def setup():
    cfg = O.OracleConfig(256, 2, 2, 64, 256, 20)          # the model of test_gpu_variants.py
    sd = O.make_state_dict(cfg, 11)
    x, text, noise = O.make_inputs(2, 40, 9, cfg, 12, steps_noise=20)
    return cfg, sd, x, text, noise


def model(cfg, sd, precision, dev):
    m = D.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=cfg.num_heads, time_dim=cfg.time_dim,
                text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps, precision=precision)
    m.load_state_dict(sd)
    return m.to(dev)


_ORACLE = {}


def oracle(setup, w, **kw):
    key = (w, tuple(sorted(kw.items())))
    if key not in _ORACLE:
        cfg, sd, x, text, noise = setup
        _ORACLE[key] = M.sample_latents_dpmpp_2m(sd, cfg, text, x, noise, w, **kw)
    return _ORACLE[key]


CASES = [dict(num_steps=k, eta=e) for e in (0.0, 1.0) for k in (5, 10, 20)] + \
        [dict(num_steps=10, eta=0.0, schedule_scale=0.3), dict(num_steps=10, eta=1.0, schedule_scale=0.3)]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kw", CASES, ids=lambda k: "-".join(f"{a}={b}" for a, b in k.items()))
@pytest.mark.parametrize("w", [5.0, None], ids=["w5", "unguided"])
@pytest.mark.parametrize("use_graph", [True, False], ids=["graph", "eager"])
def test_dpmpp_2m_vs_oracle(dev, setup, kw, w, precision, use_graph):
    cfg, sd, x, text, noise = setup
    want = oracle(setup, w, **kw)
    s = D.DiTTOSampler(model(cfg, sd, precision, dev), guidance_scale=w, method="dpmpp_2m", **kw)
    got = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise.to(dev), use_graph=use_graph)
    err = O.rel_l2(got.cpu(), want)
    assert err <= BAR[precision], err


def test_record_collects_guided_eps(dev, setup):
    cfg, sd, x, text, noise = setup
    rec_o, rec_g = [], []
    want = M.sample_latents_dpmpp_2m(sd, cfg, text, x, noise, 5.0, num_steps=5, eta=1.0, record=rec_o)
    s = D.DiTTOSampler(model(cfg, sd, "fp32", dev), guidance_scale=5.0, method="dpmpp_2m", num_steps=5, eta=1.0)
    got = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise.to(dev), record=rec_g)
    assert len(rec_g) == len(rec_o) == 5
    assert all(O.rel_l2(a.cpu(), b) <= 1e-4 for a, b in zip(rec_g, rec_o))
    assert O.rel_l2(got.cpu(), want) <= 1e-4


@pytest.mark.parametrize("use_graph", [True, False], ids=["graph", "eager"])
def test_dpmpp_2m_ragged_batch(dev, setup, use_graph):
    """2M-SDE over a sub-sequence on a mixed-length batch == every utterance sampled alone by the oracle."""
    cfg, sd, _, _, _ = setup
    g = torch.Generator().manual_seed(5)
    lengths, S_i = [24, 40, 9], [5, 9, 3]
    texts = [torch.randn(s_, cfg.text_dim, generator=g) for s_ in S_i]
    xs = [torch.randn(t_, cfg.hidden_dim, generator=g) for t_ in lengths]
    zs = [torch.randn(cfg.diffusion_steps, t_, cfg.hidden_dim, generator=g) for t_ in lengths]
    s = D.DiTTOSampler(model(cfg, sd, "fp32", dev), guidance_scale=5.0, method="dpmpp_2m", num_steps=8, eta=1.0)
    got = s.sample_latents_ragged([t.to(dev) for t in texts], lengths, x_init=[x.to(dev) for x in xs],
                                  noise=[z.to(dev) for z in zs], use_graph=use_graph)
    for i in range(3):
        want = M.sample_latents_dpmpp_2m(sd, cfg, texts[i][None], xs[i][None], zs[i][:, None], 5.0, num_steps=8, eta=1.0)
        assert O.rel_l2(got[i].cpu()[None], want) <= 1e-4


# ------------------------------------------------------------------------------------------------ the kernel
def _tables(m, steps, seed):
    """A multistep table whose even rows have c4 = 0 and the DDPM-form table with the same (c1, c2, c3), both loaded."""
    g = torch.Generator().manual_seed(seed)
    tab = torch.rand(steps, 6, generator=g) + 0.25
    tab[0::2, 3] = 0.0
    tab[1::2, 3] = -tab[1::2, 3]
    m._ensure_schedule()
    m.load_update_table(tab[:, :3].contiguous())
    m.load_multistep_table(tab)
    return tab


def test_first_order_rows_are_bit_identical_to_ddpm_update(dev, setup):
    """c4 == 0: ditto_cfg_multistep_update(_rng) gives exactly ditto_cfg_ddpm_update(_rng) with (c1, c2, c3), whatever hist held
    (NaN included); hist becomes d1 (x - d2 eps).  c4 != 0: the history term is added with one more fma."""
    cfg, sd, *_ = setup
    m = model(cfg, sd, "fp32", dev)
    steps, B, per = cfg.diffusion_steps, 3, 40 * cfg.hidden_dim
    tab = _tables(m, steps, 3)
    lib, eng = _lib.load(), m.engine()
    g = torch.Generator().manual_seed(4)
    ec, eu, x, z = (torch.randn(B, per, generator=g).to(dev) for _ in range(4))
    w = 4.0
    for t_val in (6, 7):                                   # c4 == 0, c4 != 0
        t = torch.full((B,), t_val, dtype=torch.int64, device=dev)
        ref = torch.empty_like(x)
        _lib.check(lib.ditto_cfg_ddpm_update(eng, P(ec), P(eu), P(x), P(z), P(t), w, P(ref), B, per, ST()))
        hist0 = torch.randn(B, per, generator=g).to(dev)
        for fill in (None, float("nan")):
            hist = hist0.clone() if fill is None else torch.full_like(x, fill)
            xo = x.clone()                                 # x_out aliases x
            _lib.check(lib.ditto_cfg_multistep_update(eng, P(ec), P(eu), P(xo), P(z), P(t), w, P(xo), P(hist), B, per, ST()))
            torch.cuda.synchronize()
            c1, c2, c3, c4, d1, d2 = tab[t_val].tolist()
            e64 = eu.double() + w * (ec.double() - eu.double())
            assert torch.allclose(hist.double(), d1 * (x.double() - d2 * e64), rtol=1e-5, atol=1e-5)
            if c4 == 0.0:
                assert torch.equal(xo, ref)
            elif fill is None:
                want = c1 * (x.double() - c2 * e64) + c3 * z.double() + c4 * hist0.double()
                assert torch.allclose(xo.double(), want, rtol=1e-5, atol=1e-5)
        # in-kernel noise, same {seed, draw}, no advance
        rng = torch.tensor([77, 3, 0, 0], dtype=torch.int64, device=dev)
        ref_r, out_r, hist = torch.empty_like(x), torch.empty_like(x), torch.full_like(x, float("nan"))
        _lib.check(lib.ditto_cfg_ddpm_update_rng(eng, P(ec), P(eu), P(x), P(rng), P(t), B, w, P(ref_r), B, per, 0, ST()))
        _lib.check(lib.ditto_cfg_multistep_update_rng(eng, P(ec), P(eu), P(x), P(rng), P(t), B, w, P(out_r), P(hist), B, per, 0,
                                                      ST()))
        torch.cuda.synchronize()
        if t_val == 6:
            assert torch.equal(out_r, ref_r)
        zr = torch.empty_like(x)
        _lib.check(lib.ditto_randn(P(rng), 0, P(zr), zr.numel(), ST()))
        ref_z = torch.empty_like(x)
        _lib.check(lib.ditto_cfg_ddpm_update(eng, P(ec), P(eu), P(x), P(zr), P(t), w, P(ref_z), B, per, ST()))
        torch.cuda.synchronize()
        assert torch.equal(ref_r, ref_z)                    # the drawn noise is ditto_randn's


def test_nan_history_before_first_step_is_harmless(dev, setup):
    cfg, sd, x, text, noise = setup
    s = D.DiTTOSampler(model(cfg, sd, "fp32", dev), guidance_scale=5.0, method="dpmpp_2m", num_steps=10, eta=1.0)
    xd, td, zd = x.to(dev), text.to(dev), noise.to(dev)
    a = s.sample_latents(td, x_init=xd, noise=zd)
    g = next(iter(s._graphs.values()))
    g.reset(xd, s.timesteps[0].item())
    g.hist.fill_(float("nan"))
    for t_val in s.timesteps.tolist():
        g.z.copy_(zd[t_val])
        g.t.fill_(t_val)
        g.replay()
    assert torch.equal(g.x, a) and bool(torch.isfinite(a).all())


def test_drawn_noise_equals_supplied_randn(dev, setup):
    """Graph path, eta = 1, noise drawn in the update kernel == the same job fed the ditto_randn draws of {seed, step}."""
    cfg, sd, x, text, _ = setup
    lib = _lib.load()
    s = D.DiTTOSampler(model(cfg, sd, "bf16", dev), guidance_scale=5.0, method="dpmpp_2m", num_steps=10, eta=1.0)
    xd, td = x.to(dev), text.to(dev)
    torch.manual_seed(321)
    a = s.sample_latents(td, x_init=xd)
    torch.manual_seed(321)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    noise = torch.zeros(cfg.diffusion_steps, *x.shape, device=dev)
    for k, t_val in enumerate(s.timesteps.tolist()):                 # draw k belongs to the k-th visited timestep
        rng = torch.tensor([seed, k, 0, 0], dtype=torch.int64, device=dev)
        _lib.check(lib.ditto_randn(P(rng), 0, P(noise[t_val]), noise[t_val].numel(), ST()))
    b = s.sample_latents(td, x_init=xd, noise=noise, use_graph=True)
    e = s.sample_latents(td, x_init=xd, noise=noise, use_graph=False)
    assert torch.equal(a, b) and torch.equal(a, e) and bool(torch.isfinite(a).all())


@pytest.mark.parametrize("draw", [True, False], ids=["drawn", "supplied"])
def test_launches_per_step_equal_ddim(dev, setup, draw):
    cfg, sd, x, text, noise = setup
    m = model(cfg, sd, "bf16", dev)
    counts = []
    for method in ("ddim", "dpmpp_2m"):
        s = D.DiTTOSampler(m, guidance_scale=5.0, method=method, num_steps=10)
        s.sample_latents(text.to(dev), x_init=x.to(dev), noise=None if draw else noise.to(dev))
        g = next(iter(s._graphs.values()))
        assert (g.hist is not None) == (method == "dpmpp_2m")
        counts.append(g.launches_per_step)
    assert counts[0] == counts[1] > 0


def test_three_samplers_share_one_model(dev, setup):
    """The multistep table is engine state: alternating a DDPM, a DDIM and a 2M sampler on ONE model gives each its own
    tables back."""
    cfg, sd, x, text, noise = setup
    m = model(cfg, sd, "fp32", dev)
    ref = D.DiTTOSampler(m, guidance_scale=3.0)
    ddim = D.DiTTOSampler(m, guidance_scale=3.0, method="ddim", num_steps=5)
    two = D.DiTTOSampler(m, guidance_scale=3.0, method="dpmpp_2m", num_steps=7)
    two_b = D.DiTTOSampler(m, guidance_scale=3.0, method="dpmpp_2m", num_steps=10, eta=1.0)
    xd, td, zd = x.to(dev), text.to(dev), noise.to(dev)
    first = [s.sample_latents(td, x_init=xd, noise=zd) for s in (ref, ddim, two, two_b)]
    second = [s.sample_latents(td, x_init=xd, noise=zd) for s in (two_b, two, ddim, ref)][::-1]
    for u, v in zip(first, second):
        assert torch.equal(u, v)
    assert O.rel_l2(first[0].cpu(), O.sample_latents(sd, cfg, text, x, noise, 3.0)) <= 1e-4
    assert O.rel_l2(first[1].cpu(), O.sample_latents_variant(sd, cfg, text, x, noise, 3.0, method="ddim", num_steps=5)) <= 1e-4
    assert O.rel_l2(first[2].cpu(), M.sample_latents_dpmpp_2m(sd, cfg, text, x, noise, 3.0, num_steps=7)) <= 1e-4
    assert O.rel_l2(first[3].cpu(), M.sample_latents_dpmpp_2m(sd, cfg, text, x, noise, 3.0, num_steps=10, eta=1.0)) <= 1e-4


def test_multistep_argument_checks(dev, setup):
    """Status codes, no exception across the ABI: -1 (DITTO_E_BADARG) for a wrong step count or a missing hist, -4
    (DITTO_E_STATE) without a schedule or without a multistep table.  p_sample refuses the stateful solver."""
    cfg, sd, x, text, noise = setup
    lib = _lib.load()
    steps = cfg.diffusion_steps
    tab = torch.zeros(steps, 6, device=dev)
    m = model(cfg, sd, "fp32", dev)
    eng = m.engine()
    assert lib.ditto_engine_load_multistep_table(eng, P(tab), steps, ST()) == -4          # no schedule yet
    m._ensure_schedule()
    assert lib.ditto_engine_load_multistep_table(eng, None, steps, ST()) == -1
    assert lib.ditto_engine_load_multistep_table(eng, P(tab), steps - 1, ST()) == -1
    assert b"steps" in lib.ditto_last_error()
    with pytest.raises(D.DittoError):
        m.load_multistep_table(torch.zeros(steps, 3))
    B, T, H = 1, 8, cfg.hidden_dim
    xs, eps, out, hist = (torch.zeros(B, T * H, device=dev) for _ in range(4))
    t = torch.full((B,), 3, dtype=torch.int64, device=dev)
    rng = torch.zeros(4, dtype=torch.int64, device=dev)
    assert lib.ditto_cfg_multistep_update(eng, P(eps), None, P(xs), None, P(t), 1.0, P(out), P(hist), B, T * H, ST()) == -4
    assert b"multistep table" in lib.ditto_last_error()
    assert lib.ditto_cfg_multistep_update_rng(eng, P(eps), None, P(xs), P(rng), P(t), B, 1.0, P(out), P(hist), B, T * H, 0,
                                              ST()) == -4
    ctx = m.text_context(text[:1].to(dev))
    ws = m.workspace(B, T, text.shape[1])
    e2 = torch.zeros(B, T, H, device=dev)
    assert lib.ditto_p_sample_multistep(eng, P(xs), P(ctx), P(t), None, 0, 0.0, B, T, text.shape[1], P(e2), P(out), P(hist),
                                        P(ws), ws.numel(), ST()) == -4
    assert lib.ditto_p_sample_multistep_rng(eng, P(xs), P(ctx), P(t), P(rng), 0, 0.0, B, T, text.shape[1], P(e2), P(out),
                                            P(hist), P(ws), ws.numel(), 0, ST()) == -4
    m.load_multistep_table(tab)
    assert lib.ditto_cfg_multistep_update(eng, P(eps), None, P(xs), None, P(t), 1.0, P(out), None, B, T * H, ST()) == -1
    assert lib.ditto_p_sample_multistep(eng, P(xs), P(ctx), P(t), None, 0, 0.0, B, T, text.shape[1], P(e2), P(out), None,
                                        P(ws), ws.numel(), ST()) == -1
    grp = (_lib.SeqGroup * 1)(_lib.SeqGroup(n_seq=1, n_x=1, T=T, S=text.shape[1], ctx=ctx.data_ptr()))
    assert lib.ditto_p_sample_ragged_multistep(eng, P(xs), grp, 1, P(t), None, 0, 0.0, P(e2), P(out), None, P(ws), ws.numel(),
                                               ST()) == -1
    assert lib.ditto_p_sample_ragged_multistep_rng(eng, P(xs), grp, 1, P(t), P(rng), 0, 0.0, P(e2), P(out), None, P(ws),
                                                   ws.numel(), 0, ST()) == -1
    s = D.DiTTOSampler(m, guidance_scale=3.0, method="dpmpp_2m", num_steps=5)
    with pytest.raises(D.DittoError, match="multistep"):
        s.p_sample(x.to(dev), torch.tensor([3, 3], device=dev), text.to(dev), noise=noise[3].to(dev))
