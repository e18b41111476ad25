"""Constant-text sequences (all text rows equal: the zero null embedding of the unconditional CFG half, any constant null
embedding, S = 1): their folded cross-attention output is one row per layer, which the four-CTA self-attention kernel adds
together with norm3 while the cross-attention kernel skips them.  The engine option ``no_const_text`` turns that off and is
the reference here; the oracle is the independent pin.  Bars: conditional sequences bitwise (rows do not depend on the other
sequences of the batch), unconditional ones rel-L2 <= 2e-3 against the fallback (LN3 taken in another kernel), bf16 bar
2e-2 against the oracle."""
import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from oracle import ditto_oracle as O  # checker only

pytestmark = pytest.mark.gpu
BAR, FALLBACK = 2e-2, 2e-3


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def setup(dev):
    cfg = O.OracleConfig(768, 2, 1, 256, 768, 20)
    sd = O.make_state_dict(cfg, 71)

    def build(const_text, **kw):
        m = D.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=1, time_dim=cfg.time_dim,
                    text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps, precision="bf16", **kw)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev)
        _lib.debug_option("no_const_text", 0 if const_text else 1)
        try:
            m.engine()            # engine-level option: sampled when the engine is created
        finally:
            _lib.debug_option("no_const_text", 0)
        return m

    return cfg, sd, build(True), build(False)


def rel(a, b):
    return O.rel_l2(a.float().cpu(), b.float().cpu())


def inputs(cfg, B, T, S, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, cfg.hidden_dim, generator=g)
    text = torch.randn(B, S, cfg.text_dim, generator=g)
    t = torch.randint(0, cfg.diffusion_steps, (B,), generator=g)
    return x, text, t


def guided(m, x, text, null, t, dev):
    """One CFG forward: conditional sequences first, then the unconditional ones, x shared (the sampler's layout)."""
    both = torch.cat([text, null]).to(dev)
    ctx = m.text_context(both, T_hint=x.shape[1])
    return m.forward_with_context(x.to(dev), ctx, torch.cat([t, t]).to(dev), both.shape[0], both.shape[1])


def profiled(fn):
    _lib.profile_start()
    out = fn()
    return out, _lib.profile_stop()


def test_zero_null_embedding(dev, setup):
    """C4-like shape (B = 4, T = 750, S = 64): conditional half bitwise equal to an unguided forward of the same sequences,
    unconditional half against the fallback and the oracle; the cross-attention kernel moves half the bytes."""
    cfg, sd, m, ref = setup
    B, T, S = 4, 750, 64
    x, text, t = inputs(cfg, B, T, S, 72)
    null = torch.zeros_like(text)
    out, prof = profiled(lambda: guided(m, x, text, null, t, dev))
    want, prof_ref = profiled(lambda: guided(ref, x, text, null, t, dev))
    alone = m(x.to(dev), text.to(dev), t.to(dev))
    assert torch.equal(out[:B], alone)
    assert torch.equal(out[:B], want[:B])
    assert rel(out[B:], want[B:]) <= FALLBACK, rel(out[B:], want[B:])
    for i in (0, B - 1):
        ref_u = O.ditto_forward(sd, cfg, x[i:i + 1], null[i:i + 1], t[i:i + 1])[0]
        assert rel(out[B + i], ref_u) <= BAR
    xf, xf_ref = prof["tc_gemm.cross_fused_ln"], prof_ref["tc_gemm.cross_fused_ln"]
    assert xf["launches"] == xf_ref["launches"] == cfg.num_layers
    assert xf["bytes"] == pytest.approx(xf_ref["bytes"] / 2)
    assert prof["tc_gemm.flash768_ln"]["launches"] == cfg.num_layers


def test_nonconstant_null_is_not_shortcut(dev, setup):
    cfg, sd, m, ref = setup
    x, text, t = inputs(cfg, 2, 750, 64, 73)
    null = torch.randn(text.shape, generator=torch.Generator().manual_seed(74))
    assert torch.equal(guided(m, x, text, null, t, dev), guided(ref, x, text, null, t, dev))


def test_constant_nonzero_null_and_single_token_text(dev, setup):
    cfg, sd, m, ref = setup
    B, T = 2, 750
    x, text, t = inputs(cfg, B, T, 64, 75)
    row = torch.randn(1, 1, cfg.text_dim, generator=torch.Generator().manual_seed(76))
    null = row.expand(B, 64, cfg.text_dim).contiguous()
    out, prof = profiled(lambda: guided(m, x, text, null, t, dev))
    assert prof["tc_gemm.cross_fused_ln"]["bytes"] == pytest.approx(B * T * cfg.hidden_dim * 12.0 * cfg.num_layers)
    for i in range(B):
        assert rel(out[B + i], O.ditto_forward(sd, cfg, x[i:i + 1], null[i:i + 1], t[i:i + 1])[0]) <= BAR
    # S = 1: every sequence is constant text, the conditional ones too
    x1, text1, t1 = inputs(cfg, B, T, 1, 77)
    out1, prof1 = profiled(lambda: guided(m, x1, text1, torch.zeros_like(text1), t1, dev))
    assert prof1["tc_gemm.cross_fused_ln"]["bytes"] == 0
    want1 = guided(ref, x1, text1, torch.zeros_like(text1), t1, dev)
    assert rel(out1, want1) <= FALLBACK
    for i in range(B):
        assert rel(out1[i], O.ditto_forward(sd, cfg, x1[i:i + 1], text1[i:i + 1], t1[i:i + 1])[0]) <= BAR


def test_long_text_cross_flash_kernel(dev, setup):
    """64 < S <= 256 (C3's S = 192): the cross-attention runs in flash_attn768q<CROSS>, which skips the constant items."""
    cfg, sd, m, ref = setup
    B, T, S = 2, 750, 192
    x, text, t = inputs(cfg, B, T, S, 78)
    null = torch.zeros_like(text)
    out, prof = profiled(lambda: guided(m, x, text, null, t, dev))
    want, prof_ref = profiled(lambda: guided(ref, x, text, null, t, dev))
    assert torch.equal(out[:B], want[:B])
    assert rel(out[B:], want[B:]) <= FALLBACK
    assert prof["tc_gemm.cross_flash_ln"]["bytes"] == pytest.approx(prof_ref["tc_gemm.cross_flash_ln"]["bytes"] / 2)
    assert rel(out[B], O.ditto_forward(sd, cfg, x[:1], null[:1], t[:1])[0]) <= BAR


def test_two_cta_length_keeps_the_cross_kernel(dev, setup):
    """The shortcut needs the four-CTA self-attention kernel; at a length that picks the two-CTA one (T = 300: 256-row
    tiles would pad 33 % more) the engine does not take it, and the output is bitwise the fallback's."""
    cfg, sd, m, ref = setup
    x, text, t = inputs(cfg, 2, 300, 64, 79)
    null = torch.zeros_like(text)
    assert torch.equal(guided(m, x, text, null, t, dev), guided(ref, x, text, null, t, dev))


def test_loaded_batch(dev, setup):
    """64 utterances: many items per cluster / tiles per CTA, so skipped and processed work interleave in every CTA."""
    cfg, sd, m, ref = setup
    B = 64
    x, text, t = inputs(cfg, B, 750, 64, 80)
    null = torch.zeros_like(text)
    out, want = guided(m, x, text, null, t, dev), guided(ref, x, text, null, t, dev)
    assert torch.equal(out[:B], want[:B])
    assert rel(out[B:], want[B:]) <= FALLBACK
    assert bool(torch.isfinite(out).all())


def test_ragged_cfg_sampling_on_both_cross_kernels(dev, setup):
    """Mixed lengths, CFG loop with a zero null embedding: groups on cross_fused (S <= 64) and on the CROSS flash kernel."""
    cfg, sd, m, ref = setup
    steps, w = cfg.diffusion_steps, 3.0
    lengths, text_lens = [150, 300, 150], [13, 100, 13]
    g = torch.Generator().manual_seed(81)
    xs = [torch.randn(T, cfg.hidden_dim, generator=g) for T in lengths]
    texts = [torch.randn(S, cfg.text_dim, generator=g) for S in text_lens]
    noise = [torch.randn(steps, T, cfg.hidden_dim, generator=g) for T in lengths]
    outs = {}
    for name, mm in (("fast", m), ("ref", ref)):
        s = D.DiTTOSampler(mm, guidance_scale=w)
        outs[name] = s.sample_latents_ragged([c.to(dev) for c in texts], lengths, x_init=[x.to(dev) for x in xs],
                                             noise=[z.to(dev) for z in noise], use_graph=True)
    for i in range(len(lengths)):
        assert rel(outs["fast"][i], outs["ref"][i]) <= 1e-2, (i, rel(outs["fast"][i], outs["ref"][i]))
    ref0 = O.sample_latents(sd, cfg, texts[0][None], xs[0][None], noise[0][:, None], guidance_scale=w)
    ref0 = ref0[0] if isinstance(ref0, tuple) else ref0
    assert rel(outs["fast"][0], ref0[0]) <= BAR


@pytest.mark.parametrize("method", ["ddpm", "dpmpp_2m", "known"])
def test_launches_per_step_unchanged(dev, setup, method):
    cfg, sd, m, ref = setup
    B, T = 2, 750
    x, text, _ = inputs(cfg, B, T, 64, 82)
    known_mask = torch.zeros(B, T, dtype=torch.bool)
    known_mask[:, :100] = True
    counts = []
    for mm in (m, ref):
        s = D.DiTTOSampler(mm, guidance_scale=3.0, method="ddpm" if method == "known" else method)
        kw = dict(known=x.to(dev), known_mask=known_mask.to(dev)) if method == "known" else {}
        s.sample_latents(text.to(dev), x_init=x.to(dev), **kw)
        counts.append([g.launches_per_step for g in s._graphs.values()])
    assert counts[0] == counts[1] and counts[0][0] > 0
