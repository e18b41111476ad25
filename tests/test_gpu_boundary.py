"""GPU tests (-m gpu) of the block-level boundary and the in-kernel noise:
  * GlobalAdaLN.forward / DiT.forward / RotaryEmbedding.apply_rope with the reference's signatures (src/components/DiT.py:25,61,100)
    through ditto_adaln / ditto_dit_block / ditto_rope, against the `tap::adaln` / `tap::block*` tensors the unmodified
    reference produced (tests/golden/tiny_full.npz, full_size.npz) and against the oracle;
  * ditto_randn / ditto_p_sample_rng (Philox4x32-10 + Box-Muller inside the fused update kernel) against the numpy restatement;
  * host behaviour: weight refresh, graph cache bound, timestep range checks."""
import ctypes as C

import numpy as np
import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from oracle import ditto_oracle as O  # checker only

pytestmark = pytest.mark.gpu
BAR = {"fp32": 1e-4, "bf16": 2e-2}
P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731


def ST():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def rel(a, b):
    return O.rel_l2(a.float().cpu(), b.float().cpu())


def build_model(cfg, sd, precision, dev):
    m = D.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=cfg.num_heads, time_dim=cfg.time_dim,
                text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps, precision=precision)
    m.load_state_dict(sd, strict=True)
    return m.to(dev)


def tiny(golden):
    g = golden("tiny_full.npz")
    cfg = O.OracleConfig(*[int(v) for v in g["cfg"]])
    sd = {k[4:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd::")}
    return g, cfg, sd


# ------------------------------------------------------------------------------------------ block-level signatures
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_block_level_modules_vs_reference_taps_tiny(dev, golden, precision):
    """ada_ln(x, time_embed(t_embedding(t)), text) == tap::adaln;  blocks[i](prev, text, t_emb, rotary) == tap::block{i}."""
    g, cfg, sd = tiny(golden)
    m = build_model(cfg, sd, precision, dev)
    x, text, t = (torch.from_numpy(g[k]).to(dev) for k in ("x", "text", "t"))
    t_emb = O.time_embedding(sd, torch.from_numpy(g["t"])).to(dev)          # host-side embedding MLP of DiTTO.py:75-76
    a = m.ada_ln(x, t_emb, text)
    assert rel(a, torch.from_numpy(g["tap::adaln"])) <= 1e-5                 # AdaLN is fp32 on both paths
    rot = m.rotary(x.shape[1], dev)
    assert torch.equal(rot.cpu(), torch.from_numpy(g["rotary"]))
    h = torch.from_numpy(g["tap::adaln"]).to(dev)
    for i, blk in enumerate(m.blocks):
        out = blk(h, text, t_emb, rot)                                       # the reference's call, DiTTO.py:89-90
        want = torch.from_numpy(g[f"tap::block{i}"])
        assert rel(out, want) <= BAR[precision], (i, rel(out, want))
        h = want.to(dev)
    # time_emb / rotary_pos may be omitted; a non-standard rotary table is refused, not silently ignored
    assert rel(m.blocks[0](torch.from_numpy(g["tap::adaln"]).to(dev), text), torch.from_numpy(g["tap::block0"])) <= BAR[precision]
    with pytest.raises(D.DittoError):
        m.blocks[0](h, text, t_emb, rot + 1.0)


@pytest.mark.parametrize("name", ["c1_default", "ctor_default", "ragged"])
def test_block_level_modules_vs_reference_taps_full_size(dev, golden, name):
    """Full-size configs (C1: T = 750, L = 5, one head of 768; ctor default: 12 heads of 64): AdaLN and block 0 against the
    sub-sampled taps of the unmodified reference."""
    g = golden("full_size.npz")
    H, L, heads, Td, Xd, steps, wseed, iseed, B, T, S, stride = (int(v) for v in g[f"{name}::meta"])
    cfg = O.OracleConfig(H, L, heads, Td, Xd, steps)
    sd = O.make_state_dict(cfg, wseed)
    x, text, _ = O.make_inputs(B, T, S, cfg, iseed)
    t = torch.from_numpy(g[f"{name}::t"])
    t_emb = O.time_embedding(sd, t).to(dev)
    for precision in ("fp32", "bf16"):
        m = build_model(cfg, sd, precision, dev)
        a = m.ada_ln(x.to(dev), t_emb, text.to(dev))
        assert rel(a[:, ::stride], torch.from_numpy(g[f"{name}::adaln_sub"])) <= 1e-5
        b0 = m.blocks[0](a, text.to(dev), t_emb, m.rotary(T, dev))
        e = rel(b0[:, ::stride], torch.from_numpy(g[f"{name}::block0_sub"]))
        assert e <= BAR[precision], (precision, e)


@pytest.mark.parametrize("hidden,heads,T,S", [(768, 1, 130, 20), (256, 4, 77, 9)])
def test_standalone_dit_block_and_adaln_vs_oracle(dev, hidden, heads, T, S):
    """components/DiT.py modules constructed on their own (no DiTTO around them): a private blocks-only engine."""
    torch.manual_seed(7)
    blk = D.DiT(hidden, heads, 64, hidden).to(dev)
    ada = D.GlobalAdaLN(hidden, 64, hidden).to(dev)
    sd = {"blocks.0." + k: v.detach().cpu() for k, v in blk.state_dict().items()}
    sd.update({"ada_ln." + k: v.detach().cpu() for k, v in ada.state_dict().items()})
    g = torch.Generator().manual_seed(8)
    x, text, te = torch.randn(2, T, hidden, generator=g), torch.randn(2, S, hidden, generator=g), torch.randn(2, 64, generator=g)
    want_a = O.global_adaln(sd, x, te, text)
    assert rel(ada(x.to(dev), te.to(dev), text.to(dev)), want_a) <= 1e-5
    want_b = O.dit_block(sd, 0, x, text, O.rotary_angles(T, hidden // heads), heads)
    got = blk(x.to(dev), text.to(dev), te.to(dev), blk.rotary(T, dev))
    assert rel(got, want_b) <= BAR["bf16"]
    # in-place weight edit + refresh: the engine follows
    with torch.no_grad():
        blk.mlp_fc2.bias.data.add_(1.0)
    blk._own.refresh_weights()
    sd["blocks.0.mlp_fc2.bias"] = sd["blocks.0.mlp_fc2.bias"] + 1.0
    assert rel(blk(x.to(dev), text.to(dev)), O.dit_block(sd, 0, x, text, O.rotary_angles(T, hidden // heads), heads)) <= BAR["bf16"]


def test_blocks_only_engine_refuses_the_whole_model_calls(dev):
    """A stand-alone block's engine (DITTO_F_BLOCKS_ONLY) holds no proj_in, t embedding or AdaLN weights: even with a schedule
    loaded, the ragged forward and sampler calls return DITTO_E_STATE and launch nothing."""
    torch.manual_seed(9)
    blk = D.DiT(256, 4, 64, 256).to(dev)
    x, text = torch.randn(1, 8, 256, device=dev), torch.randn(1, 3, 256, device=dev)
    blk(x, text)                                                    # builds the block's engine
    lib, eng = _lib.load(), blk._own.engine()
    half = torch.full((1,), 0.5, device=dev)                        # betas, alphas, alphas_cumprod of its one step
    assert lib.ditto_engine_load_schedule(eng, P(half), P(half), P(half), 1, ST()) == 0
    torch.cuda.synchronize()
    buf = torch.zeros(1 << 20, device=dev)                           # stands in for every buffer: nothing may touch it
    t = torch.zeros(1, dtype=torch.int64, device=dev)
    grp = (_lib.SeqGroup * 1)(_lib.SeqGroup(n_seq=1, n_x=1, T=8, S=3, ctx=buf.data_ptr()))
    n0 = _lib.launch_count()
    assert lib.ditto_forward_ragged(eng, P(x), grp, 1, P(t), P(buf), P(buf), buf.numel() * 4, ST()) == -4
    assert lib.ditto_p_sample_ragged(eng, P(x), grp, 1, P(t), P(buf), 0, 0.0, P(buf), P(buf), P(buf), buf.numel() * 4, ST()) == -4
    assert lib.ditto_p_sample_ragged_multistep(eng, P(x), grp, 1, P(t), P(buf), 0, 0.0, P(buf), P(buf), P(buf), P(buf),
                                               buf.numel() * 4, ST()) == -4
    assert b"blocks-only" in lib.ditto_last_error()
    assert _lib.launch_count() == n0
    torch.cuda.synchronize()
    assert not bool(buf.any())


@pytest.mark.parametrize("b,T,h,d", [(2, 24, 2, 32), (1, 750, 1, 768), (3, 5, 12, 64)])
def test_apply_rope_vs_oracle(dev, b, T, h, d):
    g = torch.Generator().manual_seed(3)
    t = torch.randn(b, T, h, d, generator=g)
    rot = D.RotaryEmbedding(d).to(dev)
    pos = rot(T, dev)
    assert torch.equal(pos.cpu(), O.rotary_angles(T, d))
    assert rel(rot.apply_rope(pos, t.to(dev)), O.apply_rope(pos.cpu(), t)) <= 2e-6
    with pytest.raises(D.DittoError):
        rot.apply_rope(pos[:, :-2], t.to(dev))


# ------------------------------------------------------------------------------------------ in-kernel noise
def rng_state(seed, draw, dev):
    return torch.tensor([seed, draw, 0, 0], dtype=torch.int64, device=dev)


@pytest.mark.parametrize("seed,draw,n,off", [(1234, 0, 4096, 0), (2 ** 61 + 17, 49, 1003, 8), (0, 2 ** 33, 17, 4 * (2 ** 31))])
def test_randn_matches_philox_restatement(dev, seed, draw, n, off):
    lib = _lib.load()
    out = torch.empty(n + 3, device=dev)[:n]
    _lib.check(lib.ditto_randn(P(rng_state(seed, draw, dev)), off, P(out), n, ST()))
    want = O.philox_normal(seed, draw, n, off)
    # same Philox bits; the Box-Muller transform uses the MUFU log2 / sin / cos approximations (abs error ~1e-6 of |z| <= 6)
    assert float((out.cpu() - want).abs().max()) <= 2e-5


def test_randn_statistics_and_streams(dev):
    lib = _lib.load()
    n = 1 << 22
    z = torch.empty(n, device=dev)
    _lib.check(lib.ditto_randn(P(rng_state(5, 0, dev)), 0, P(z), n, ST()))
    zz = z.double()
    assert abs(float(zz.mean())) < 3e-3 and abs(float(zz.var()) - 1.0) < 5e-3
    assert abs(float((zz ** 4).mean()) - 3.0) < 0.03 and abs(float((zz ** 3).mean())) < 0.02
    assert abs(float((zz[:-1] * zz[1:]).mean())) < 3e-3                  # neighbours uncorrelated
    z2 = torch.empty(n, device=dev)
    _lib.check(lib.ditto_randn(P(rng_state(5, 1, dev)), 0, P(z2), n, ST()))     # next draw: a different stream
    assert abs(float((zz * z2.double()).mean())) < 3e-3 and not torch.equal(z, z2)
    _lib.check(lib.ditto_randn(P(rng_state(5, 0, dev)), 0, P(z2), n, ST()))     # same (seed, draw): the same numbers
    assert torch.equal(z, z2)


@pytest.mark.parametrize("guided", [True, False])
def test_p_sample_rng_equals_p_sample_with_the_same_noise(dev, guided):
    """ditto_p_sample_rng == ditto_p_sample fed with z = ditto_randn(seed, draw): bit for bit; `advance` decrements every t and
    bumps the draw counter (the bookkeeping of SpeechGenerator.py:161-162)."""
    lib = _lib.load()
    cfg = O.OracleConfig(256, 2, 1, 64, 256, 10)
    sd = O.make_state_dict(cfg, 5)
    m = build_model(cfg, sd, "bf16", dev)
    s = D.DiTTOSampler(m, guidance_scale=2.5 if guided else None)
    B, T, S = 3, 40, 7
    x, text, _ = O.make_inputs(B, T, S, cfg, 6)
    xd = x.to(dev)
    n = 2 * B if guided else B
    ctx = s._context(text.to(dev), guided, None, T)
    ws = m.workspace(n, T, S)
    eps = torch.empty(n, T, 256, device=dev)
    t = torch.full((n,), 7, dtype=torch.int64, device=dev)
    rng = rng_state(99, 3, dev)
    z = torch.empty_like(xd)
    _lib.check(lib.ditto_randn(P(rng), 0, P(z), z.numel(), ST()))
    want = torch.empty_like(xd)
    s._p_sample_raw(xd, ctx, t, z, guided, 2.5 if guided else 0.0, S, eps, want, ws=ws)
    got = torch.empty_like(xd)
    _lib.check(lib.ditto_p_sample_rng(m.engine(), P(xd), P(ctx), P(t), P(rng), 1 if guided else 0, 2.5 if guided else 0.0, B, T, S,
                                      P(eps), P(got), P(ws), ws.numel(), 1, ST()))
    assert torch.equal(got, want)
    assert t.tolist() == [6] * n and rng.tolist() == [99, 4, 0, 0]
    _lib.check(lib.ditto_p_sample_rng(m.engine(), P(xd), P(ctx), P(t), P(rng), 1 if guided else 0, 2.5 if guided else 0.0, B, T, S,
                                      P(eps), P(got), P(ws), ws.numel(), 0, ST()))
    assert t.tolist() == [6] * n and rng.tolist() == [99, 4, 0, 0]      # advance = 0 leaves the bookkeeping alone
    assert not torch.equal(got, want)                                   # other t, other draw


def test_graph_sampling_with_internal_noise_is_reproducible_and_matches_eager(dev):
    """sample_latents (CUDA-graph replay, noise drawn in the update kernel) == the eager loop fed with the same Philox draws;
    torch.manual_seed makes a sampling job repeatable; two jobs without reseeding differ."""
    lib = _lib.load()
    cfg = O.OracleConfig(256, 2, 1, 64, 256, 12)
    sd = O.make_state_dict(cfg, 15)
    m = build_model(cfg, sd, "bf16", dev)
    s = D.DiTTOSampler(m, guidance_scale=3.0)
    B, T, S = 2, 33, 6
    x, text, _ = O.make_inputs(B, T, S, cfg, 16)
    torch.manual_seed(123)
    a = s.sample_latents(text.to(dev), x_init=x.to(dev))
    b = s.sample_latents(text.to(dev), x_init=x.to(dev))
    torch.manual_seed(123)
    c = s.sample_latents(text.to(dev), x_init=x.to(dev))
    assert torch.equal(a, c) and not torch.equal(a, b) and bool(torch.isfinite(a).all())
    torch.manual_seed(123)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    noise = torch.empty(cfg.diffusion_steps, B, T, 256, device=dev)
    for k, t_val in enumerate(reversed(range(cfg.diffusion_steps))):    # draw k belongs to timestep steps - 1 - k
        _lib.check(lib.ditto_randn(P(rng_state(seed, k, dev)), 0, P(noise[t_val]), noise[t_val].numel(), ST()))
    e = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise, use_graph=False)
    assert torch.equal(a, e)
    # the captured step holds kernels of this library only: its launch count equals the library's own counter
    g = next(iter(s._graphs.values()))
    assert g.launches_per_step > 0 and g.z is None


def test_ragged_graph_with_internal_noise_is_cached_and_reproducible(dev):
    cfg = O.OracleConfig(256, 2, 1, 64, 256, 6)
    sd = O.make_state_dict(cfg, 25)
    m = build_model(cfg, sd, "bf16", dev)
    s = D.DiTTOSampler(m, guidance_scale=2.0)
    gen = torch.Generator().manual_seed(26)
    lengths, tl = [20, 33, 20, 9], [4, 7, 4, 2]
    texts = [torch.randn(k, 256, generator=gen).to(dev) for k in tl]
    xs = [torch.randn(k, 256, generator=gen).to(dev) for k in lengths]
    torch.manual_seed(9)
    a = s.sample_latents_ragged(texts, lengths, x_init=xs)
    assert len(s._ragged_graphs) == 1
    torch.manual_seed(9)
    b = s.sample_latents_ragged(texts, lengths, x_init=xs)
    assert len(s._ragged_graphs) == 1                                   # same signature: graph re-used, not re-captured
    for u, v in zip(a, b):
        assert torch.equal(u, v) and bool(torch.isfinite(u).all())
    texts2 = [t * 0.5 for t in texts]                                   # same shapes, other content: cached graph, new contexts
    torch.manual_seed(9)
    c = s.sample_latents_ragged(texts2, lengths, x_init=xs)
    e = s.sample_latents_ragged(texts2, lengths, x_init=xs, use_graph=False,
                                noise=None)                             # eager path draws with torch: only finiteness / shape
    assert len(s._ragged_graphs) == 1 and not torch.equal(a[1], c[1])
    assert all(tuple(u.shape) == tuple(v.shape) for u, v in zip(c, e))


# ------------------------------------------------------------------------------------------ host behaviour
def test_weight_edits_and_refresh(dev):
    cfg = O.OracleConfig(128, 1, 2, 32, 128, 5)
    sd = O.make_state_dict(cfg, 31)
    m = build_model(cfg, sd, "fp32", dev)
    x, text, _ = O.make_inputs(1, 16, 4, cfg, 32)
    t = torch.tensor([2])
    base = m(x.to(dev), text.to(dev), t.to(dev))
    with torch.no_grad():
        m.proj_out.bias.add_(1.0)                     # versioned in-place edit: picked up automatically
    assert rel(m(x.to(dev), text.to(dev), t.to(dev)), base.cpu() + 1.0) <= 1e-6
    m.proj_out.bias.data.add_(1.0)                    # .data edit: invisible to the version counter ...
    stale = m(x.to(dev), text.to(dev), t.to(dev))
    assert rel(stale, base.cpu() + 1.0) <= 1e-6
    m.refresh_weights()                               # ... until the documented refresh
    assert rel(m(x.to(dev), text.to(dev), t.to(dev)), base.cpu() + 2.0) <= 1e-6


def test_step_graph_cache_is_bounded(dev):
    cfg = O.OracleConfig(128, 1, 2, 32, 128, 4)
    m = build_model(cfg, O.make_state_dict(cfg, 33), "bf16", dev)
    s = D.DiTTOSampler(m, guidance_scale=3.0)
    s.max_cached_graphs = 2
    g = torch.Generator().manual_seed(34)
    for T in (8, 9, 10, 8):
        text, x = torch.randn(1, 3, 128, generator=g).to(dev), torch.randn(1, T, 128, generator=g).to(dev)
        assert bool(torch.isfinite(s.sample_latents(text, x_init=x)).all())
        assert len(s._graphs) <= 2
    assert [k[1] for k in s._graphs] == [10, 8]


def test_out_of_range_timesteps_raise(dev):
    cfg = O.OracleConfig(128, 1, 2, 32, 128, 5)
    m = build_model(cfg, O.make_state_dict(cfg, 35), "fp32", dev)
    x, text, _ = O.make_inputs(1, 8, 3, cfg, 36)
    for bad in (5, -1):
        with pytest.raises(D.DittoError):
            m(x.to(dev), text.to(dev), torch.tensor([bad]).to(dev))
        with pytest.raises(D.DittoError):
            m.q_sample(x.to(dev), torch.tensor([bad]).to(dev))
        with pytest.raises(D.DittoError):
            D.DiTTOSampler(m).p_sample(x.to(dev), torch.tensor([bad]).to(dev), text.to(dev))


REMOVED_OPTIONS = ["no_mcast", "no_fused_ln", "dbg_nostore", "cluster_m", "cluster_n", "stages_1cta", "stages_pair", "xf_prefetch",
                   "pv_transpose", "rope_table", "no_rope_fast32", "no_pair", "generic_epi", "no_fused_attn"]
KEPT_OPTIONS = ["no_flash", "no_flash768", "no_fused_cross", "no_cross_flash", "no_const_text", "no_fc2_ln", "flash768_quad",
                "rope_generic", "glu_generic", "no_pv_perm4", "xf_rows", "side_streams", "defer_ln2", "no_defer_ln"]


def test_debug_options_are_explicit(dev):
    lib = _lib.load()
    assert lib.ditto_debug_option(b"no_such_option", 1) == -1
    try:
        for name in REMOVED_OPTIONS:
            assert lib.ditto_debug_option(name.encode(), 1) == -1, name
        for name in KEPT_OPTIONS:
            assert lib.ditto_debug_option(name.encode(), 0) == 0, name
    finally:
        _lib.debug_option("reset", 0)
    # ditto_attn_self768 defines flag bit 0 only: any other bit is refused before a kernel is launched
    n, T, H = 1, 64, 768
    qkv = torch.zeros(n * T, 3 * H, dtype=torch.bfloat16, device=dev)
    hh = torch.zeros(n * T, H, device=dev)
    u = torch.zeros(n * T, H, dtype=torch.bfloat16, device=dev)
    gamma, beta = torch.ones(H, device=dev), torch.zeros(H, device=dev)
    args = (P(qkv), 3 * H, n, T, 0.125, P(hh), P(gamma), P(beta), P(u))
    before = lib.ditto_kernel_launch_count()
    assert lib.ditto_attn_self768(*args, 1 << 16, ST()) == -1
    assert lib.ditto_kernel_launch_count() == before
    _lib.check(lib.ditto_attn_self768(*args, 1, ST()), "ditto_attn_self768")   # the same buffers with a defined flag run
    torch.cuda.synchronize()
    assert lib.ditto_kernel_launch_count() > before
