"""GPU checks of sampling around known frames (speech prompt, infilling) through the C-ABI (ditto_engine_load_known_table +
ditto_p_sample_known and friends): parity with the textbook replacement sampler of oracle/known_ref.py, the kernel's pins to
the plain update kernels, in-kernel noise, launch counts, table ownership between samplers, and the status codes."""
import ctypes as C

import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from oracle import ditto_oracle as O
from oracle import known_ref as KR

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
    """The model and inputs of test_gpu_multistep.py with four utterances: a 12-frame prompt, a span 15:30 to fill, no known
    frame, every frame known."""
    cfg = O.OracleConfig(256, 2, 2, 64, 256, 20)
    sd = O.make_state_dict(cfg, 11)
    x, text, noise = O.make_inputs(4, 40, 9, cfg, 12, steps_noise=20)
    known = torch.randn(4, 40, cfg.hidden_dim, generator=torch.Generator().manual_seed(13))
    mask = torch.zeros(4, 40, dtype=torch.bool)
    mask[0, :12] = True
    mask[1] = True
    mask[1, 15:30] = False
    mask[3] = True
    return cfg, sd, x, text, noise, known, mask


def model(cfg, sd, precision, dev):
    m = D.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=cfg.num_heads, time_dim=cfg.time_dim,
                text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps, precision=precision)
    m.load_state_dict(sd)
    return m.to(dev)


_ORACLE = {}


def oracle(setup, w, kw):
    key = (w, tuple(sorted(kw.items())))
    if key not in _ORACLE:
        cfg, sd, x, text, noise, known, mask = setup
        _ORACLE[key] = KR.sample_latents_known(sd, cfg, text, x, noise, known, mask, w, **kw)
    return _ORACLE[key]


CASES = [dict(method="ddpm"), dict(method="ddim", num_steps=10), dict(method="dpmpp_2m", num_steps=10),
         dict(method="dpmpp_2m", num_steps=10, eta=1.0), dict(method="ddim", num_steps=10, eta=1.0, schedule_scale=0.3),
         dict(method="dpmpp_2m", num_steps=10, eta=1.0, schedule_scale=0.3)]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kw", CASES, ids=lambda k: "-".join(f"{a}={b}" for a, b in k.items()))
@pytest.mark.parametrize("w", [5.0, None], ids=["w5", "unguided"])
@pytest.mark.parametrize("use_graph", [True, False], ids=["graph", "eager"])
def test_known_frames_vs_oracle(dev, setup, kw, w, precision, use_graph):
    cfg, sd, x, text, noise, known, mask = setup
    want = oracle(setup, w, kw)
    s = D.DiTTOSampler(model(cfg, sd, precision, dev), guidance_scale=w, **kw)
    got = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise.to(dev), use_graph=use_graph, known=known.to(dev),
                           known_mask=mask.to(dev))
    err = O.rel_l2(got.cpu(), want)
    assert err <= BAR[precision], err
    assert torch.equal(got.cpu()[mask], known[mask])          # the known frames come back exactly


def test_record_collects_guided_eps(dev, setup):
    cfg, sd, x, text, noise, known, mask = setup
    kw = dict(method="dpmpp_2m", num_steps=5, eta=1.0)
    rec_o, rec_g = [], []
    want = KR.sample_latents_known(sd, cfg, text, x, noise, known, mask, 5.0, record=rec_o, **kw)
    s = D.DiTTOSampler(model(cfg, sd, "fp32", dev), guidance_scale=5.0, **kw)
    got = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise.to(dev), record=rec_g, known=known.to(dev),
                           known_mask=mask.to(dev))
    assert len(rec_g) == len(rec_o) == 5
    assert all(O.rel_l2(a.cpu(), b) <= 1e-4 for a, b in zip(rec_g, rec_o))
    assert O.rel_l2(got.cpu(), want) <= 1e-4


@pytest.mark.parametrize("kw", [dict(method="ddpm"), dict(method="ddim", num_steps=10, eta=1.0),
                                dict(method="dpmpp_2m", num_steps=10, eta=1.0)], ids=["ddpm", "ddim", "2m"])
def test_all_false_mask_is_the_unprompted_job(dev, setup, kw):
    """Bit-identical to the job without known frames: supplied noise (graph, eager), drawn noise with the same seed (graph)
    and the same generator (eager)."""
    cfg, sd, x, text, noise, known, _ = setup
    s = D.DiTTOSampler(model(cfg, sd, "bf16", dev), guidance_scale=5.0, **kw)
    xd, td, zd, kd = x.to(dev), text.to(dev), noise.to(dev), known.to(dev)
    none = torch.zeros(4, 40, dtype=torch.bool, device=dev)
    for use_graph in (True, False):
        a = s.sample_latents(td, x_init=xd, noise=zd, use_graph=use_graph)
        b = s.sample_latents(td, x_init=xd, noise=zd, use_graph=use_graph, known=kd, known_mask=none)
        assert torch.equal(a, b)
    torch.manual_seed(5)
    a = s.sample_latents(td, x_init=xd)
    torch.manual_seed(5)
    b = s.sample_latents(td, x_init=xd, known=kd, known_mask=none)
    assert torch.equal(a, b)
    a = s.sample_latents(td, x_init=xd, generator=torch.Generator(device=dev).manual_seed(6))
    b = s.sample_latents(td, x_init=xd, generator=torch.Generator(device=dev).manual_seed(6), known=kd, known_mask=none)
    assert torch.equal(a, b) and bool(torch.isfinite(a).all())


# ------------------------------------------------------------------------------------------------ the kernel
def _tables(m, steps, seed):
    """Random DDPM-form, multistep (c4 != 0 on odd rows) and known tables, all loaded."""
    g = torch.Generator().manual_seed(seed)
    tab = torch.rand(steps, 6, generator=g) + 0.25
    tab[0::2, 3] = 0.0
    tab[1::2, 3] = -tab[1::2, 3]
    kt = torch.rand(steps, 2, generator=g) + 0.25
    m._ensure_schedule()
    m.load_update_table(tab[:, :3].contiguous())
    m.load_multistep_table(tab)
    m.load_known_table(kt)
    return tab, kt


def test_update_kernel_pins(dev, setup):
    """Unknown frames: bit-identical to ditto_cfg_ddpm_update(_rng) / ditto_cfg_multistep_update(_rng), hist included.  Known
    frames: a p + s z (drawn z == ditto_randn at the same offsets), hist untouched, and NaN in eps, x and hist there does not
    reach the output."""
    cfg, sd, *_ = setup
    m = model(cfg, sd, "fp32", dev)
    steps, B, T, H = cfg.diffusion_steps, 3, 40, cfg.hidden_dim
    per = T * H
    _, kt = _tables(m, steps, 3)
    lib, eng = _lib.load(), m.engine()
    g = torch.Generator().manual_seed(4)
    ec, eu, x, z, p = (torch.randn(B, per, generator=g).to(dev) for _ in range(5))
    hist0 = torch.randn(B, per, generator=g).to(dev)
    mask = torch.zeros(B, T, dtype=torch.uint8)
    mask[0, :9] = 1
    mask[1, 17:33] = 1
    mask = mask.to(dev)
    kn = mask.bool().repeat_interleave(H, dim=1)                      # [B, per] element mask
    poison = lambda v: torch.where(kn, torch.full_like(v, float("nan")), v)   # noqa: E731
    ecn, eun, xn = poison(ec), poison(eu), poison(x)
    w = 4.0
    rng = torch.tensor([77, 3, 0, 0], dtype=torch.int64, device=dev)
    zr = torch.empty_like(x)
    _lib.check(lib.ditto_randn(P(rng), 0, P(zr), zr.numel(), ST()))
    for t_val in (6, 7):                                   # c4 == 0, c4 != 0
        t = torch.full((B,), t_val, dtype=torch.int64, device=dev)
        a, s_ = kt[t_val].tolist()
        for multistep in (False, True):
            for draw in (False, True):
                ref, out = torch.empty_like(x), torch.empty_like(x)
                h_ref, h_out = hist0.clone(), poison(hist0)
                if multistep and draw:
                    _lib.check(lib.ditto_cfg_multistep_update_rng(eng, P(ec), P(eu), P(x), P(rng), P(t), B, w, P(ref), P(h_ref), B, per,
                                                                  0, ST()))
                elif multistep:
                    _lib.check(lib.ditto_cfg_multistep_update(eng, P(ec), P(eu), P(x), P(z), P(t), w, P(ref), P(h_ref), B, per, ST()))
                elif draw:
                    _lib.check(lib.ditto_cfg_ddpm_update_rng(eng, P(ec), P(eu), P(x), P(rng), P(t), B, w, P(ref), B, per, 0, ST()))
                else:
                    _lib.check(lib.ditto_cfg_ddpm_update(eng, P(ec), P(eu), P(x), P(z), P(t), w, P(ref), B, per, ST()))
                _lib.check(lib.ditto_cfg_update_known(eng, P(ecn), P(eun), P(xn), None if draw else P(z), P(rng) if draw else None,
                                                      P(t), B, w, P(out), P(h_out) if multistep else None, P(p), P(mask), B, T, 0,
                                                      ST()))
                torch.cuda.synchronize()
                assert torch.equal(out[~kn], ref[~kn]), (t_val, multistep, draw)
                zz = zr if draw else z
                want = a * p[kn].double() + s_ * zz[kn].double()
                assert torch.allclose(out[kn].double(), want, rtol=1e-6, atol=1e-6), (t_val, multistep, draw)
                assert bool(torch.isfinite(out).all())
                if multistep:
                    assert torch.equal(h_out[~kn], h_ref[~kn])
                    assert bool(torch.isnan(h_out[kn]).all())          # known frames leave hist as it was
    # x_out aliasing x, and the last visited row {1, 0} returns p exactly
    m.load_known_table(torch.tensor([[1.0, 0.0]]).expand(steps, 2).contiguous())
    t = torch.full((B,), 0, dtype=torch.int64, device=dev)
    xo = x.clone()
    _lib.check(lib.ditto_cfg_update_known(eng, P(ec), P(eu), P(xo), None, P(rng), P(t), B, w, P(xo), None, P(p), P(mask), B, T, 0, ST()))
    torch.cuda.synchronize()
    assert torch.equal(xo[kn], p[kn])


def test_advance_bookkeeping(dev, setup):
    """advance: the draw counter goes up by one and every t[i < n_t] down by one, as with ditto_cfg_ddpm_update_rng."""
    cfg, sd, *_ = setup
    m = model(cfg, sd, "fp32", dev)
    _tables(m, cfg.diffusion_steps, 5)
    lib, eng = _lib.load(), m.engine()
    B, T, H = 2, 40, cfg.hidden_dim
    ec, x, p = (torch.randn(B, T * H, device=dev) for _ in range(3))
    mask = torch.zeros(B, T, dtype=torch.uint8, device=dev)
    mask[:, :5] = 1
    out = torch.empty_like(x)
    rng = torch.tensor([9, 4, 0, 0], dtype=torch.int64, device=dev)
    t = torch.tensor([7, 7, 7, 7], dtype=torch.int64, device=dev)
    _lib.check(lib.ditto_cfg_update_known(eng, P(ec), None, P(x), None, P(rng), P(t), 4, 1.0, P(out), None, P(p), P(mask), B, T, 1, ST()))
    torch.cuda.synchronize()
    assert rng.tolist() == [9, 5, 0, 0] and t.tolist() == [6, 6, 6, 6]


def test_drawn_noise_equals_supplied_randn(dev, setup):
    """Graph path, noise drawn in the update kernel == the same job fed the ditto_randn draws of {seed, step}, on the graph
    and the eager path."""
    cfg, sd, x, text, _, known, mask = setup
    lib = _lib.load()
    s = D.DiTTOSampler(model(cfg, sd, "bf16", dev), guidance_scale=5.0, method="dpmpp_2m", num_steps=10, eta=1.0)
    xd, td, kd, md = x.to(dev), text.to(dev), known.to(dev), mask.to(dev)
    torch.manual_seed(321)
    a = s.sample_latents(td, x_init=xd, known=kd, known_mask=md)
    torch.manual_seed(321)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    noise = torch.zeros(cfg.diffusion_steps, *x.shape, device=dev)
    for k, t_val in enumerate(s.timesteps.tolist()):                 # draw k belongs to the k-th visited timestep
        rng = torch.tensor([seed, k, 0, 0], dtype=torch.int64, device=dev)
        _lib.check(lib.ditto_randn(P(rng), 0, P(noise[t_val]), noise[t_val].numel(), ST()))
    b = s.sample_latents(td, x_init=xd, noise=noise, use_graph=True, known=kd, known_mask=md)
    e = s.sample_latents(td, x_init=xd, noise=noise, use_graph=False, known=kd, known_mask=md)
    assert torch.equal(a, b) and torch.equal(a, e) and bool(torch.isfinite(a).all())
    assert torch.equal(a[md], kd[md])


@pytest.mark.parametrize("draw", [True, False], ids=["drawn", "supplied"])
@pytest.mark.parametrize("method", ["ddim", "dpmpp_2m"])
def test_launches_per_step_equal_unprompted(dev, setup, draw, method):
    cfg, sd, x, text, noise, known, mask = setup
    s = D.DiTTOSampler(model(cfg, sd, "bf16", dev), guidance_scale=5.0, method=method, num_steps=10)
    z = None if draw else noise.to(dev)
    s.sample_latents(text.to(dev), x_init=x.to(dev), noise=z)
    s.sample_latents(text.to(dev), x_init=x.to(dev), noise=z, known=known.to(dev), known_mask=mask.to(dev))
    graphs = list(s._graphs.values())
    assert len(graphs) == 2 and graphs[0].known is None and graphs[1].known is not None
    assert graphs[0].launches_per_step == graphs[1].launches_per_step > 0


@pytest.mark.parametrize("use_graph", [True, False], ids=["graph", "eager"])
def test_ragged_batch(dev, setup, use_graph):
    """Three utterances of different lengths and prompt lengths == each sampled alone by the oracle."""
    cfg, sd, *_ = setup
    g = torch.Generator().manual_seed(5)
    lengths, S_i, prompts = [24, 40, 9], [5, 9, 3], [6, 15, 0]
    texts = [torch.randn(s_, cfg.text_dim, generator=g) for s_ in S_i]
    xs = [torch.randn(t_, cfg.hidden_dim, generator=g) for t_ in lengths]
    zs = [torch.randn(cfg.diffusion_steps, t_, cfg.hidden_dim, generator=g) for t_ in lengths]
    ps = [torch.randn(t_, cfg.hidden_dim, generator=g) for t_ in lengths]
    ms = [torch.arange(t_) < p_ for t_, p_ in zip(lengths, prompts)]
    ms[2][3:6] = True                                   # the shortest one: a kept span instead of a prompt
    kw = dict(method="dpmpp_2m", num_steps=8, eta=1.0)
    s = D.DiTTOSampler(model(cfg, sd, "fp32", dev), guidance_scale=5.0, **kw)
    got = s.sample_latents_ragged([t.to(dev) for t in texts], lengths, x_init=[x.to(dev) for x in xs],
                                  noise=[z.to(dev) for z in zs], use_graph=use_graph, known=[p.to(dev) for p in ps],
                                  known_mask=[q.to(dev) for q in ms])
    for i in range(3):
        want = KR.sample_latents_known(sd, cfg, texts[i][None], xs[i][None], zs[i][:, None], ps[i][None], ms[i][None], 5.0, **kw)
        assert O.rel_l2(got[i].cpu()[None], want) <= 1e-4
        assert torch.equal(got[i].cpu()[ms[i]], ps[i][ms[i]])
    if use_graph:     # noise drawn in the per-group kernels: the known frames still come back exactly
        out = s.sample_latents_ragged([t.to(dev) for t in texts], lengths, x_init=[x.to(dev) for x in xs],
                                      known=[p.to(dev) for p in ps], known_mask=[q.to(dev) for q in ms])
        for i in range(3):
            assert torch.equal(out[i].cpu()[ms[i]], ps[i][ms[i]]) and bool(torch.isfinite(out[i]).all())


def test_samplers_share_one_model(dev, setup):
    """The known table is engine state: alternating samplers with different schedules on ONE model gives each its own table
    back, also after q_sample re-loaded the module's schedule."""
    cfg, sd, x, text, noise, known, mask = setup
    m = model(cfg, sd, "fp32", dev)
    kws = [dict(), dict(method="ddim", num_steps=5), dict(method="dpmpp_2m", num_steps=7, schedule_scale=0.3)]
    ss = [D.DiTTOSampler(m, guidance_scale=3.0, **kw) for kw in kws]
    xd, td, zd, kd, md = x.to(dev), text.to(dev), noise.to(dev), known.to(dev), mask.to(dev)
    first = [s.sample_latents(td, x_init=xd, noise=zd, known=kd, known_mask=md) for s in ss]
    m.q_sample(xd, torch.full((4,), 3, dtype=torch.int64, device=dev), zd[0])    # the module's schedule, owner None again
    second = [None] * 3
    for i in (0, 2, 1):    # the reference sampler first: its schedule is loaded, the known table is the 2M sampler's
        second[i] = ss[i].sample_latents(td, x_init=xd, noise=zd, known=kd, known_mask=md)
    for u, v, kw in zip(first, second, kws):
        assert torch.equal(u, v)
        want = KR.sample_latents_known(sd, cfg, text, x, noise, known, mask, 3.0, **({"method": "ddpm"} | kw))
        assert O.rel_l2(u.cpu(), want) <= 1e-4


def test_argument_checks(dev, setup):
    """Status codes, no exception across the ABI: -4 (DITTO_E_STATE) without a known table, -1 (DITTO_E_BADARG) for both or
    neither of z / rng, a mask without latents and advance with supplied noise; the Python API validates its inputs."""
    cfg, sd, x, text, noise, known, mask = setup
    lib = _lib.load()
    steps = cfg.diffusion_steps
    m = model(cfg, sd, "fp32", dev)
    eng = m.engine()
    kt = torch.zeros(steps, 2, device=dev)
    assert lib.ditto_engine_load_known_table(eng, P(kt), steps, ST()) == -4          # no schedule yet
    m._ensure_schedule()
    assert lib.ditto_engine_load_known_table(eng, None, steps, ST()) == -1
    assert lib.ditto_engine_load_known_table(eng, P(kt), steps - 1, ST()) == -1
    assert b"steps" in lib.ditto_last_error()
    with pytest.raises(D.DittoError):
        m.load_known_table(torch.zeros(steps, 3))
    B, T, H = 1, 8, cfg.hidden_dim
    xs, eps, out, z, p = (torch.zeros(B, T * H, device=dev) for _ in range(5))
    mk = torch.ones(B, T, dtype=torch.uint8, device=dev)
    t = torch.full((B,), 3, dtype=torch.int64, device=dev)
    rng = torch.zeros(4, dtype=torch.int64, device=dev)
    ctx = m.text_context(text[:1].to(dev))
    ws = m.workspace(B, T, text.shape[1])
    e2 = torch.zeros(B, T, H, device=dev)
    grp = (_lib.SeqGroup * 1)(_lib.SeqGroup(n_seq=1, n_x=1, T=T, S=text.shape[1], ctx=ctx.data_ptr()))

    def upd(z_, r_, known_, mask_, adv=0):
        return lib.ditto_cfg_update_known(eng, P(eps), None, P(xs), z_, r_, P(t), B, 1.0, P(out), None, known_, mask_, B, T, adv, ST())

    def ps(z_, r_, known_, mask_, adv=0):
        return lib.ditto_p_sample_known(eng, P(xs), P(ctx), P(t), z_, r_, 0, 0.0, B, T, text.shape[1], P(e2), P(out), None, known_,
                                        mask_, P(ws), ws.numel(), adv, ST())

    def pr(z_, r_, known_, mask_, adv=0):
        return lib.ditto_p_sample_ragged_known(eng, P(xs), grp, 1, P(t), z_, r_, 0, 0.0, P(e2), P(out), None, known_, mask_, P(ws),
                                               ws.numel(), adv, ST())

    for call in (upd, ps, pr):
        assert call(P(z), None, P(p), P(mk)) == -4                                    # no known table loaded
        assert b"known table" in lib.ditto_last_error()
    m.load_known_table(kt)
    for call in (upd, ps, pr):
        assert call(P(z), P(rng), P(p), P(mk)) == -1                                  # both z and rng
        assert call(None, None, P(p), P(mk)) == -1                                    # neither
        assert call(P(z), None, None, P(mk)) == -1                                    # a mask without latents
        assert call(P(z), None, P(p), None) == -1                                     # latents without a mask
        assert call(P(z), None, P(p), P(mk), adv=1) == -1                             # advance with supplied noise
        assert b"advance" in lib.ditto_last_error()
    hist = torch.zeros(B, T * H, device=dev)
    assert lib.ditto_cfg_update_known(eng, P(eps), None, P(xs), P(z), None, P(t), B, 1.0, P(out), P(hist), P(p), P(mk), B, T, 0,
                                      ST()) == -4                                     # hist without a multistep table
    assert b"multistep table" in lib.ditto_last_error()
    # the Python API
    s = D.DiTTOSampler(m, guidance_scale=3.0)
    xd, td, kd, md = x.to(dev), text.to(dev), known.to(dev), mask.to(dev)
    for bad in (dict(known=kd), dict(known_mask=md), dict(known=kd[:, :20], known_mask=md), dict(known=kd, known_mask=md[:, :20]),
                dict(known=kd.double(), known_mask=md), dict(known=kd, known_mask=md.float()), dict(known=known, known_mask=md),
                dict(known=kd, known_mask=mask)):
        with pytest.raises(D.DittoError):
            s.sample_latents(td, x_init=xd, **bad)
    with pytest.raises(D.DittoError):
        s.sample_latents_ragged([td[0]], [40], known=[kd[0]])
