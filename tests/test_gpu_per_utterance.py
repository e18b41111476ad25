"""GPU checks of per-utterance seeds and guidance scales (ditto_p_sample_per_utt, ditto_p_sample_ragged_per_utt,
ditto_cfg_update_per_utt, ditto_randn_latents; sample_latents(_ragged)(..., seeds=, guidance_scale=[...])).

  * the noise stream: utterance b's draw k is ditto_randn({s_b, k}, 0, T H) bit for bit, and x_T is its draw 2^64 - 1, at
    every position of a uniform and of a ragged batch; observed through the update kernel with an update table of rows
    {0, 0, 1}, where x_out = z exactly;
  * per-utterance w: one update with w = [w_0 .. w_B-1] is, row by row and bitwise, B updates with the scalar w_b;
  * graph == eager == the eager loop fed the same noise, bitwise, for every sampler, with and without known frames;
  * an utterance's result does not depend on its batch-mates beyond the forward's batch-dependent rounding;
  * one captured graph serves every scale;
  * bad arguments come back as DITTO_E_BADARG."""
import ctypes as C
import random

import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from ditto_tts_b200.parallel import c5_lengths
from ditto_tts_b200.ragged import RaggedBatch
from ditto_tts_b200.sampler import randn_latents
from oracle import ditto_oracle as O  # checker only

pytestmark = pytest.mark.gpu
E_BADARG = -1
XT_DRAW = 2 ** 64 - 1
CFG = O.OracleConfig(256, 2, 2, 64, 256, 10)
SEEDS = [7, 2 ** 64 - 1, 123456789012345, 7, 2 ** 63 + 5]   # equal seeds at positions 0 and 3; both halves of the uint64 range


def P(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def ST():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def i64(v):
    return v - 2 ** 64 if v >= 2 ** 63 else v


def seeds_dev(seeds, dev):
    return torch.tensor([i64(s) for s in seeds], dtype=torch.int64, device=dev)


def rng_state(seed, draw, dev):
    return torch.tensor([i64(seed), i64(draw), 0, 0], dtype=torch.int64, device=dev)


def randn(seed, draw, n, dev):
    """ditto_randn({seed, draw}, elem_offset 0, n): the utterance's noise by the contract."""
    out = torch.empty(n, device=dev)
    rng = rng_state(seed, draw, dev)    # held until the launch: a freed temporary's block can be handed out again before it
    _lib.check(_lib.load().ditto_randn(P(rng), 0, P(out), n, ST()))
    return out


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def build_model(cfg, sd, precision, dev):
    m = D.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=cfg.num_heads, time_dim=cfg.time_dim,
                text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps, precision=precision)
    m.load_state_dict(sd, strict=True)
    return m.to(dev)


@pytest.fixture(scope="module")
def sd():
    return O.make_state_dict(CFG, 31)


@pytest.fixture(scope="module")
def zmodel(sd, dev):
    """A model whose update table has rows {0, 0, 1} (x_out = z): the noise the kernel uses, observed exactly."""
    m = build_model(CFG, sd, "bf16", dev)
    s = D.DiTTOSampler(m, 2.0)
    m.load_update_table(torch.tensor([[0.0, 0.0, 1.0]] * CFG.diffusion_steps))
    return m, s


# ------------------------------------------------------------------------------------------------ the noise stream
@pytest.mark.parametrize("draw", [0, 3, 2 ** 40 + 1])
def test_uniform_step_noise_is_each_utterances_own_stream(dev, zmodel, draw):
    zmodel, s = zmodel
    B, T, S, H = len(SEEDS), 12, 5, CFG.hidden_dim
    x, text, _ = O.make_inputs(B, T, S, CFG, 3)
    ctx = s._context(text.to(dev), True, None, T)
    t = torch.full((2 * B,), 4, dtype=torch.int64, device=dev)
    eps = torch.empty(2 * B, T, H, device=dev)
    out = torch.empty(B, T, H, device=dev)
    rng = rng_state(99, draw, dev)
    ws = zmodel.workspace(2 * B, T, S)
    x_dev, sdv = x.to(dev), seeds_dev(SEEDS, dev)   # locals, alive until the kernel has read them
    _lib.check(_lib.load().ditto_p_sample_per_utt(zmodel.engine(), P(x_dev), P(ctx), P(t), None, P(rng), P(sdv), 1, 2.0, None, B, T, S,
                                                  P(eps), P(out), None, None, None, P(ws), ws.numel(), 0, ST()))
    for b, sb in enumerate(SEEDS):
        want = randn(sb, draw, T * H, dev)
        assert torch.equal(out[b].flatten(), want), b
        assert float((out[b].flatten().cpu() - O.philox_normal(sb, draw, T * H)).abs().max()) <= 2e-5
    assert torch.equal(out[0], out[3])                                   # equal seeds, different positions
    assert float(rng[1]) == draw                                         # advance = 0: the draw counter stays


def test_ragged_step_noise_is_each_utterances_own_stream(dev, zmodel):
    """Several groups, the utterances of a group at several positions: packed-group seeds offset per group by the engine."""
    zmodel = zmodel[0]
    lengths, tokens = [12, 20, 12, 7, 20, 12], [5, 3, 5, 9, 3, 4]
    seeds = [5, 2 ** 64 - 2, 11, 5, 3, 2 ** 63]
    g = torch.Generator().manual_seed(4)
    texts = [torch.randn(k, CFG.text_dim, generator=g).to(dev) for k in tokens]
    rb = RaggedBatch(zmodel, texts, lengths, guided=True)
    assert len(rb.groups) == 4
    x = torch.randn(rb.x_rows, CFG.hidden_dim, generator=g).to(dev)
    t = torch.full((rb.n_seq,), 2, dtype=torch.int64, device=dev)
    eps = torch.empty(rb.seq_rows, CFG.hidden_dim, device=dev)
    out = torch.empty_like(x)
    rng = rng_state(1, 6, dev)
    rb.p_sample(x, t, None, 0.0, eps, out, rng=rng, seeds=rb.pack_seeds(seeds), w_dev=rb.pack_w([1.0] * 6), advance=False)
    per = rb.unpack(out)
    for i, sb in enumerate(seeds):
        assert torch.equal(per[i].flatten(), randn(sb, 6, lengths[i] * CFG.hidden_dim, dev)), i
    assert torch.equal(per[0][:7], per[3])                               # same seed, other group: the same leading normals
    # x_T: one launch over the packed rows, each utterance's reserved draw
    xt = rb.unpack(randn_latents(rb.pack_seeds(seeds), rb.row0(), rb.x_rows, CFG.hidden_dim))
    for i, sb in enumerate(seeds):
        want = randn(sb, XT_DRAW, lengths[i] * CFG.hidden_dim, dev)
        assert torch.equal(xt[i].flatten(), want), i
        assert float((xt[i].flatten().cpu() - O.philox_normal(sb, XT_DRAW, lengths[i] * CFG.hidden_dim)).abs().max()) <= 2e-5


def test_uniform_x_T_and_independence(dev):
    B, T, H = len(SEEDS), 64, 256
    sdv = seeds_dev(SEEDS, dev)
    xt = randn_latents(sdv, torch.arange(0, (B + 1) * T, T, dtype=torch.int64, device=dev), B * T, H).view(B, T, H)
    for b, sb in enumerate(SEEDS):
        assert torch.equal(xt[b].flatten(), randn(sb, XT_DRAW, T * H, dev)), b
    assert torch.equal(xt[0], xt[3])
    flat = xt.flatten(1).double()
    n = flat.shape[1]
    for a, b in [(0, 1), (0, 2), (1, 4), (2, 4)]:                        # different seeds: uncorrelated (|r| < 5 / sqrt(n))
        r = float(torch.corrcoef(flat[[a, b]])[0, 1])
        assert abs(r) < 5 / n ** 0.5, (a, b, r)
    # the reserved draw is not a step draw
    assert not torch.equal(xt[0].flatten(), randn(SEEDS[0], 0, T * H, dev))


# ------------------------------------------------------------------------------------------------ per-utterance w
FORMS = ["ddpm", "multistep", "known"]


@pytest.mark.parametrize("noise", ["z", "seeds"])
@pytest.mark.parametrize("form", FORMS)
def test_per_utterance_w_equals_scalar_runs(dev, sd, form, noise):
    """Row b of one update with w = [w_0 .. w_B-1] == the update with the scalar w_b, bitwise (same eps, x, z / seeds)."""
    m = build_model(CFG, sd, "bf16", dev)
    kw = dict(method="dpmpp_2m", num_steps=5) if form == "multistep" else {}
    s = D.DiTTOSampler(m, 1.0, **kw)
    s._activate(known=form == "known")
    B, T, H = 4, 16, CFG.hidden_dim
    ws_ = [0.5, 3.0, 7.25, -1.0]
    g = torch.Generator().manual_seed(8)
    ec, eu, x, z, hist0, known = (torch.randn(B, T, H, generator=g).to(dev) for _ in range(6))
    mask = (torch.rand(B, T, generator=g) < 0.3).to(torch.uint8).to(dev) if form == "known" else None
    tv = int(s.timesteps[2])                              # a second-order row of the multistep table
    if form == "multistep":
        assert float(s.multistep_table[tv, 3]) != 0.0
    lib = _lib.load()

    def run(w_scalar, w_vec):
        t = torch.full((B,), tv, dtype=torch.int64, device=dev)
        out = torch.empty_like(x)
        hist = hist0.clone() if form == "multistep" else None
        rng = rng_state(0, 2, dev) if noise == "seeds" else None
        sdv = seeds_dev(SEEDS[:B], dev) if noise == "seeds" else None
        _lib.check(lib.ditto_cfg_update_per_utt(m.engine(), P(ec), P(eu), P(x), P(z) if noise == "z" else None, P(rng), P(sdv),
                                                P(t), B, w_scalar, P(w_vec), P(out), P(hist), P(known) if mask is not None else None,
                                                P(mask), B, T, 0, ST()))
        return out, hist

    got, ghist = run(0.0, torch.tensor(ws_, device=dev))
    for b, wb in enumerate(ws_):
        want, whist = run(wb, None)
        assert torch.equal(got[b], want[b]), b
        if ghist is not None:
            assert torch.equal(ghist[b], whist[b]), b


# ------------------------------------------------------------------------------------------------ graph vs eager
SAMPLERS = [dict(method="ddpm"), dict(method="ddim", num_steps=5), dict(method="dpmpp_2m", num_steps=5)]
SID = ["ddpm", "ddim5", "dpmpp2m5"]


def noise_for(s, seeds, lengths, H, dev):
    """noise[t] per utterance = ditto_randn({s_b, k}, 0) for the k-th visited timestep t; x_T = the reserved draw."""
    steps = s.model.diffusion_steps
    zs, xs = [], []
    for sb, T in zip(seeds, lengths):
        z = torch.zeros(steps, T, H, device=dev)
        for k, tv in enumerate(s.timesteps.tolist()):
            z[tv] = randn(sb, k, T * H, dev).view(T, H)
        zs.append(z)
        xs.append(randn(sb, XT_DRAW, T * H, dev).view(T, H))
    return zs, xs


@pytest.mark.parametrize("known", [False, True], ids=["plain", "known"])
@pytest.mark.parametrize("kw", SAMPLERS, ids=SID)
def test_uniform_seeded_graph_equals_eager_and_fed_noise(dev, sd, kw, known):
    m = build_model(CFG, sd, "bf16", dev)
    s = D.DiTTOSampler(m, 2.0, **kw)
    B, T, S, H = 3, 24, 6, CFG.hidden_dim
    seeds, w = SEEDS[:B], [0.0, 2.5, 6.0]
    _, text, _ = O.make_inputs(B, T, S, CFG, 21)
    text = text.to(dev)
    shape = torch.empty(B, T, H, device=dev)
    kk = {}
    if known:
        g = torch.Generator().manual_seed(22)
        mask = torch.zeros(B, T, dtype=torch.bool)
        mask[:, :6] = True
        kk = dict(known=torch.randn(B, T, H, generator=g).to(dev), known_mask=mask.to(dev))
    a = s.sample_latents(text, shape, seeds=seeds, guidance_scale=w, **kk)
    b = s.sample_latents(text, shape, seeds=seeds, guidance_scale=w, **kk)
    c = s.sample_latents(text, shape, seeds=seeds, guidance_scale=w, use_graph=False, **kk)
    zs, xs = noise_for(s, seeds, [T] * B, H, dev)
    d = s.sample_latents(text, x_init=torch.stack(xs), noise=torch.stack(zs, dim=1), guidance_scale=w, use_graph=False, **kk)
    assert torch.isfinite(a).all()
    assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(a, d)


@pytest.mark.parametrize("known", [False, True], ids=["plain", "known"])
@pytest.mark.parametrize("kw", SAMPLERS, ids=SID)
def test_ragged_seeded_graph_equals_eager_and_fed_noise(dev, sd, kw, known):
    m = build_model(CFG, sd, "bf16", dev)
    s = D.DiTTOSampler(m, 2.0, **kw)
    lengths, tokens = [20, 12, 20, 9], [4, 6, 4, 3]
    seeds, w = [3, 2 ** 64 - 9, 3, 17], [1.0, 4.0, 2.5, 0.0]
    g = torch.Generator().manual_seed(23)
    texts = [torch.randn(k, CFG.text_dim, generator=g).to(dev) for k in tokens]
    kk = {}
    if known:
        kk = dict(known=[torch.randn(T, CFG.hidden_dim, generator=g).to(dev) for T in lengths],
                  known_mask=[(torch.arange(T) < 5).to(dev) for T in lengths])
    a = s.sample_latents_ragged(texts, lengths, seeds=seeds, guidance_scale=w, **kk)
    b = s.sample_latents_ragged(texts, lengths, seeds=seeds, guidance_scale=w, **kk)
    c = s.sample_latents_ragged(texts, lengths, seeds=seeds, guidance_scale=w, use_graph=False, **kk)
    zs, xs = noise_for(s, seeds, lengths, CFG.hidden_dim, dev)
    d = s.sample_latents_ragged(texts, lengths, x_init=xs, noise=zs, guidance_scale=w, use_graph=False, **kk)
    for i in range(len(lengths)):
        assert torch.isfinite(a[i]).all()
        assert torch.equal(a[i], b[i]) and torch.equal(a[i], c[i]) and torch.equal(a[i], d[i]), i


# ------------------------------------------------------------------------------------------------ batch composition
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_result_does_not_depend_on_batch_mates(dev, precision):
    """C5-mix lengths in shuffled order, seeds and mixed w: every utterance against the same utterance sampled alone, and the
    batch against its two halves run one after the other (what sharding does).  The noise and x_T are identical by
    construction; what could be left is the forward's batch-dependent rounding.

    Measured on a B200 (1000 W; DDIM, 8 steps of 50, H = 768, 2 layers, these ten C5 lengths): none, in either precision.
    Every utterance of the batch, of the two halves, alone in a ragged batch and alone as a uniform [1, T, H] job came out
    bitwise equal: the GEMMs reduce every output row over K in one fixed order whatever the number of rows (no split-K, no
    atomics), attention and the AdaLN / RoPE tables are per sequence, and the update is element-wise.  So equality is
    asserted, and any reduction order that starts to depend on the batch shows up here."""
    cfg = O.OracleConfig(768, 2, 1, 256, 768, 50)
    m = build_model(cfg, O.make_state_dict(cfg, 41), precision, dev)
    s = D.DiTTOSampler(m, 3.0, method="ddim", num_steps=8)
    T_all, S_all = c5_lengths(256)
    pick = list(range(0, 256, 23))[:10]
    rnd = random.Random(5)
    rnd.shuffle(pick)
    T, Sx = [T_all[i] for i in pick], [S_all[i] for i in pick]
    g = torch.Generator().manual_seed(42)
    texts = [torch.randn(k, cfg.text_dim, generator=g).to(dev) for k in Sx]
    seeds = [rnd.randrange(2 ** 64) for _ in pick]
    w = [rnd.choice([1.0, 2.0, 3.0, 5.0]) for _ in pick]
    full = s.sample_latents_ragged(texts, T, seeds=seeds, guidance_scale=w)
    h = len(pick) // 2
    halves = (s.sample_latents_ragged(texts[:h], T[:h], seeds=seeds[:h], guidance_scale=w[:h]) +
              s.sample_latents_ragged(texts[h:], T[h:], seeds=seeds[h:], guidance_scale=w[h:]))
    alone = [s.sample_latents_ragged([texts[i]], [T[i]], seeds=[seeds[i]], guidance_scale=[w[i]])[0] for i in range(len(pick))]
    # the uniform layout: the same utterance as a [1, T, H] job
    uni = s.sample_latents(texts[0][None], torch.empty(1, T[0], cfg.hidden_dim, device=dev), seeds=[seeds[0]], guidance_scale=[w[0]])[0]
    errs = [max(O.rel_l2(full[i].cpu(), alone[i].cpu()), O.rel_l2(halves[i].cpu(), alone[i].cpu())) for i in range(len(pick))]
    e_uni = O.rel_l2(uni.cpu(), alone[0].cpu())
    bitwise = all(torch.equal(full[i], alone[i]) and torch.equal(halves[i], alone[i]) for i in range(len(pick)))
    assert bitwise and torch.equal(uni, alone[0]), (errs, e_uni)


# ------------------------------------------------------------------------------------------------ graph reuse
@pytest.mark.parametrize("ragged", [False, True], ids=["uniform", "ragged"])
def test_one_graph_serves_every_scale(dev, sd, ragged):
    m = build_model(CFG, sd, "bf16", dev)
    s = D.DiTTOSampler(m, 2.0, method="ddim", num_steps=5)
    B, T, S, H = 3, 16, 5, CFG.hidden_dim
    seeds = SEEDS[:B]
    g = torch.Generator().manual_seed(24)
    texts = [torch.randn(S + i, CFG.text_dim, generator=g).to(dev) for i in range(B)]
    lengths = [T, T + 4, T]
    text_u = torch.randn(B, S, CFG.text_dim, generator=g).to(dev)
    shape = torch.empty(B, T, H, device=dev)

    def job(w, use_graph=True, **kw):
        if ragged:
            return torch.cat(s.sample_latents_ragged(texts, lengths, guidance_scale=w, use_graph=use_graph, **kw))
        return s.sample_latents(text_u, shape, guidance_scale=w, use_graph=use_graph, **kw)

    x0 = torch.randn(B, T, H, generator=g).to(dev)
    xr = [torch.randn(Ti, H, generator=g).to(dev) for Ti in lengths]
    for w in (2.0, 5.0, [1.0, 3.0, 6.0], 0.5):
        got = job(w, seeds=seeds)
        assert torch.equal(got, job(w, seeds=seeds, use_graph=False)), w
        # unseeded with supplied x_T: the graph of scalar jobs, now fed from the scale buffer, against the eager scalar path
        xin = xr if ragged else x0
        zs = ([torch.randn(CFG.diffusion_steps, Ti, H, generator=g).to(dev) for Ti in lengths] if ragged else
              torch.randn(CFG.diffusion_steps, B, T, H, generator=g).to(dev))
        assert torch.equal(job(w, x_init=xin, noise=zs), job(w, x_init=xin, noise=zs, use_graph=False)), w
    # one seeded and one supplied-noise graph for all four scales (a graph per scale would have filled the 4-entry cache)
    if ragged:
        assert len(s._ragged_graphs) == 1 and len(next(iter(s._ragged_graphs.values()))[1]) == 2
    else:
        assert len(s._graphs) == 2


# ------------------------------------------------------------------------------------------------ rejections
def test_bad_arguments_are_badarg(dev, sd):
    m = build_model(CFG, sd, "bf16", dev)
    s = D.DiTTOSampler(m, 2.0)
    s._activate()
    lib = _lib.load()
    B, T, S, H = 2, 8, 3, CFG.hidden_dim
    x = torch.zeros(B, T, H, device=dev)
    z = torch.zeros_like(x)
    t = torch.full((2 * B,), 3, dtype=torch.int64, device=dev)
    rng = rng_state(1, 0, dev)
    sdv = seeds_dev([1, 2], dev)
    out = torch.empty_like(x)
    eps = torch.empty(2 * B, T, H, device=dev)
    ctx = s._context(torch.zeros(B, S, CFG.text_dim, device=dev), True, None, T)
    ws = m.workspace(2 * B, T, S)

    def upd(zz, rr, ss):
        return lib.ditto_cfg_update_per_utt(m.engine(), P(x), P(x), P(x), P(zz), P(rr), P(ss), P(t), B, 1.0, None, P(out), None, None,
                                            None, B, T, 0, ST())

    def step(zz, rr, ss):
        return lib.ditto_p_sample_per_utt(m.engine(), P(x), P(ctx), P(t), P(zz), P(rr), P(ss), 1, 1.0, None, B, T, S, P(eps), P(out),
                                          None, None, None, P(ws), ws.numel(), 0, ST())

    for call in (upd, step):
        assert call(None, None, sdv) == E_BADARG and b"seeds need rng" in lib.ditto_last_error()
        assert call(z, None, sdv) == E_BADARG and b"seeds and z" in lib.ditto_last_error()
        assert call(z, rng, sdv) == E_BADARG
        assert call(None, rng, sdv) == 0
    rb = RaggedBatch(m, [torch.zeros(S, CFG.text_dim, device=dev)] * B, [T] * B, guided=True)
    assert lib.ditto_p_sample_ragged_per_utt(m.engine(), P(x), rb.c_groups, len(rb.groups), P(t), None, None, P(sdv), 1, 1.0, None,
                                             P(eps), P(out), None, None, None, P(rb.workspace()), rb.workspace().numel(), 0,
                                             ST()) == E_BADARG
    row0 = torch.tensor([0, T, 2 * T], dtype=torch.int64, device=dev)
    assert lib.ditto_randn_latents(None, P(row0), B, H, P(out), ST()) == E_BADARG
    assert lib.ditto_randn_latents(P(sdv), None, B, H, P(out), ST()) == E_BADARG
    assert lib.ditto_randn_latents(P(sdv), P(row0), B, H - 2, P(out), ST()) == E_BADARG
    torch.cuda.synchronize()
    # host side
    shape = torch.empty(B, T, H, device=dev)
    text = torch.zeros(B, S, CFG.text_dim, device=dev)
    for kw in (dict(seeds=[1]), dict(seeds=[1, 2 ** 64]), dict(seeds=[-1, 2]), dict(seeds=[1, 2], noise=torch.zeros(10, B, T, H, device=dev)),
               dict(seeds=[1, 2], generator=torch.Generator(device=dev)), dict(guidance_scale=[1.0]),
               dict(guidance_scale=[1.0, float("nan")])):
        with pytest.raises(D.DittoError):
            s.sample_latents(text, shape, **kw)
    with pytest.raises(D.DittoError):
        s.sample_latents_ragged([text[0], text[1]], [T, T], seeds=[1, 2, 3])
