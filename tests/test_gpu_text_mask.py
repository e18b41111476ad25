"""Per-utterance text lengths (ditto_text_context_masked, ``text_lengths=``): texts of different token counts padded to one
width S_pad.  Sequence i must compute what it computes alone with the unpadded text[:len], whatever the padded rows hold.

Every cross-attention path is covered.  The folded kernels (cross_fused for S <= 64, flash_attn768q<CROSS> for 64 < S <= 256,
the folded scores GEMM or the fused scores kernel with a bias, softmax and P.V) see the mask as a -inf score bias.  The
unfolded ones (multi-head, single head above S = 384, no folding) and the fp32 path read the per-sequence valid key count
from the context."""
import ctypes as C

import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from oracle import ditto_oracle as O  # checker only

pytestmark = pytest.mark.gpu
BAR = {"bf16": 2e-2, "fp32": 1e-4}
SAME_KERNEL_ROW = 1e-5

# name -> (hidden, heads, precision, engine switches, DiTTO keywords, T, S_pad, lengths, lengths whose unpadded run takes the
# kernel S_pad takes).  Every case has a one-token text (constant text with padding).
CASES = {
    "cross_fused": (768, 1, "bf16", {}, {}, 750, 64, [64, 40, 9, 1], [64, 40, 9, 1]),
    "cross_flash": (768, 1, "bf16", {}, {}, 750, 192, [192, 150, 65, 30, 1], [192, 150, 65]),
    "folded_scores_300": (768, 1, "bf16", {}, {}, 150, 300, [300, 280, 100, 1], [300, 280]),
    "unfolded_two_tile_512": (768, 1, "bf16", {}, {}, 150, 512, [512, 400, 200, 1], [512, 400]),
    "multihead_folded": (256, 4, "bf16", {}, {}, 150, 24, [24, 17, 1], [24, 17, 1]),
    "multihead_unfolded": (256, 4, "bf16", {}, {}, 150, 48, [48, 40, 20, 1], [48, 40]),
    "fp32": (768, 1, "fp32", {}, {}, 150, 64, [64, 30, 1], [64, 30, 1]),
    "no_fused_cross": (768, 1, "bf16", {"no_fused_cross": 1}, {}, 150, 64, [64, 33, 1], [64, 33, 1]),
    "no_cross_flash": (768, 1, "bf16", {"no_cross_flash": 1}, {}, 150, 192, [192, 100, 1], [192, 100]),
    "unfused_softmax_400": (768, 1, "bf16", {}, {"fused_attn": False}, 150, 400, [400, 390, 1], [400, 390]),
}


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


_models = {}


def model(name, dev):
    """(cfg, sd, module) of a case, engine created under the case's switches (engine-level options are sampled then)."""
    H, heads, prec, opts, kw = CASES[name][:5]
    key = (H, heads, prec, tuple(sorted(opts.items())), tuple(sorted(kw.items())))
    if key not in _models:
        cfg = O.OracleConfig(H, 2, heads, 256, H, 20)
        sd = O.make_state_dict(cfg, 91 + H + heads)
        m = D.DiTTO(hidden_dim=H, num_layers=2, num_heads=heads, time_dim=256, text_dim=H, diffusion_steps=20, precision=prec, **kw)
        m.load_state_dict(sd, strict=True)
        m = m.to(dev)
        for k, v in opts.items():
            _lib.debug_option(k, v)
        try:
            m.engine()
        finally:
            _lib.debug_option("reset", 0)
        _models[key] = (cfg, sd, m)
    return _models[key]


def inputs(cfg, B, T, S, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, cfg.hidden_dim, generator=g)
    text = torch.randn(B, S, cfg.text_dim, generator=g)
    t = torch.randint(0, cfg.diffusion_steps, (B,), generator=g)
    return x, text, t


def fill_padding(text, lens, how):
    out = text.clone()
    g = torch.Generator().manual_seed(7)
    for i, n in enumerate(lens):
        rows = out[i, n:]
        if how == "zeros":
            rows.zero_()
        elif how == "randn":
            rows.copy_(torch.randn(rows.shape, generator=g))
        elif how == "big":
            rows.fill_(1e4)
        else:
            rows.copy_(torch.randn(rows.shape, generator=g))
            rows[..., 0::2] = float("nan")
            rows[..., 1::4] = float("inf")
            rows[..., 3::4] = float("-inf")
    return out


def rel(a, b):
    return O.rel_l2(a.double().cpu(), b.double().cpu())


def row_rel(a, b):
    a, b = a.double().cpu().reshape(-1, a.shape[-1]), b.double().cpu().reshape(-1, b.shape[-1])
    return float(((a - b).norm(dim=1) / b.norm(dim=1).clamp_min(1e-30)).max())


def f64(sd):
    return {k: v.double() for k, v in sd.items()}


@pytest.mark.parametrize("name", list(CASES))
def test_pad_content_is_invisible(dev, name):
    cfg, sd, m = model(name, dev)
    T, S, lens = CASES[name][5:8]
    x, text, t = inputs(cfg, len(lens), T, S, 100)
    outs = [m(x.to(dev), fill_padding(text, lens, how).to(dev), t.to(dev), text_lengths=lens)
            for how in ("zeros", "randn", "big", "nan_inf")]
    assert bool(torch.isfinite(outs[0]).all())
    for o in outs[1:]:
        assert torch.equal(o, outs[0])


@pytest.mark.parametrize("name", list(CASES))
def test_full_length_mask_is_the_plain_context(dev, name):
    cfg, sd, m = model(name, dev)
    T, S, lens = CASES[name][5:8]
    x, text, t = inputs(cfg, len(lens), T, S, 101)
    xd, td, tt = x.to(dev), text.to(dev), t.to(dev)
    plain = m(xd, td, tt)
    assert torch.equal(m(xd, td, tt, text_lengths=[S] * len(lens)), plain)
    # a full-length sequence of a masked batch is the plain one too (rows do not depend on their batch-mates)
    assert lens[0] == S and torch.equal(m(xd, td, tt, text_lengths=lens)[0], plain[0])


@pytest.mark.parametrize("name", list(CASES))
def test_mask_equals_the_shorter_text(dev, name):
    cfg, sd, m = model(name, dev)
    prec = CASES[name][2]
    T, S, lens, same = CASES[name][5:9]
    x, text, t = inputs(cfg, len(lens), T, S, 102)
    out = m(x.to(dev), fill_padding(text, lens, "randn").to(dev), t.to(dev), text_lengths=lens)
    sd64 = f64(sd)
    for i, n in enumerate(lens):
        if n in same:
            alone = m(x[i:i + 1].to(dev), text[i:i + 1, :n].contiguous().to(dev), t[i:i + 1].to(dev))[0]
            assert row_rel(out[i], alone) <= SAME_KERNEL_ROW, (i, n, row_rel(out[i], alone))
        want = O.ditto_forward(sd64, cfg, x[i:i + 1].double(), text[i:i + 1, :n].double(), t[i:i + 1])[0]
        assert rel(out[i], want) <= BAR[prec], (i, n, rel(out[i], want))


@pytest.mark.parametrize("name", ["cross_fused", "cross_flash", "unfolded_two_tile_512", "multihead_folded", "multihead_unfolded", "fp32"])
def test_attn_cross_against_oracle(dev, name):
    """ditto_attn_cross (the cross-attention section alone) reads the masked context like the whole forward."""
    cfg, sd, m = model(name, dev)
    prec = CASES[name][2]
    T, S, lens = CASES[name][5:8]
    B = len(lens)
    x, text, _ = inputs(cfg, B, T, S, 103)
    text = fill_padding(text, lens, "nan_inf")
    xd = x.to(dev)
    ctx = m.text_context(text.to(dev), name="block_ctx", T_hint=T, text_lengths=lens)
    out = torch.empty_like(xd)
    ws = m.workspace(B, T, S)
    _lib.check(_lib.load().ditto_attn_cross(m.engine(), 0, C.c_void_p(xd.data_ptr()), C.c_void_p(ctx.data_ptr()), B, T, S,
                                            C.c_void_p(out.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream)), "ditto_attn_cross")
    sd64 = f64(sd)
    for i, n in enumerate(lens):
        want = O.cross_attention(sd64, "blocks.0.", x[i:i + 1].double(), text[i:i + 1, :n].double(), cfg.num_heads)[0]
        # the increment (section output - x) is what the section computes; the residual would hide it
        assert rel(out[i] - xd[i], want - x[i].double()) <= BAR[prec], (i, n)


# ------------------------------------------------------------------------------------------------ sampling
SAMPLE_KW = {"ddpm": dict(), "dpmpp_2m": dict(method="dpmpp_2m", num_steps=8)}


def _known(B, T, H, dev):
    g = torch.Generator().manual_seed(5)
    mask = torch.zeros(B, T, dtype=torch.bool)
    mask[:, :40] = True
    return torch.randn(B, T, H, generator=g).to(dev), mask.to(dev)


@pytest.mark.parametrize("method,known,use_graph", [("ddpm", False, True), ("ddpm", False, False), ("dpmpp_2m", False, True),
                                                    ("ddpm", True, True)])
def test_uniform_sampling_equals_each_unpadded_text(dev, method, known, use_graph):
    cfg, sd, m = model("cross_fused", dev)
    s = D.DiTTOSampler(m, 3.0, **SAMPLE_KW[method])
    B, T, S, lens, seeds = 3, 150, 64, [64, 23, 1], [11, 12, 13]
    _, text, _ = inputs(cfg, B, T, S, 104)
    text = fill_padding(text, lens, "nan_inf").to(dev)
    shape = torch.empty(B, T, cfg.hidden_dim, device=dev)
    kw = {}
    if known:
        kp, km = _known(B, T, cfg.hidden_dim, dev)
        kw = dict(known=kp, known_mask=km)
    out = s.sample_latents(text, shape, seeds=seeds, text_lengths=lens, use_graph=use_graph, **kw)
    assert bool(torch.isfinite(out).all())
    for i, n in enumerate(lens):
        kwi = {k: v[i:i + 1] for k, v in kw.items()}
        alone = s.sample_latents(text[i:i + 1, :n].contiguous(), shape[i:i + 1], seeds=[seeds[i]], use_graph=use_graph, **kwi)[0]
        assert rel(out[i], alone) <= SAME_KERNEL_ROW, (i, n, rel(out[i], alone))
    # an utterance's result does not depend on its batch-mates' lengths
    other = s.sample_latents(text, shape, seeds=seeds, text_lengths=[64, 5, 1], use_graph=use_graph, **kw)
    assert torch.equal(other[0], out[0]) and torch.equal(other[2], out[2])


@pytest.mark.parametrize("method,known,use_graph", [("ddpm", False, True), ("ddpm", False, False), ("dpmpp_2m", False, True),
                                                    ("ddpm", True, True)])
def test_ragged_sampling_equals_each_unpadded_text(dev, method, known, use_graph):
    cfg, sd, m = model("cross_flash", dev)
    s = D.DiTTOSampler(m, 3.0, **SAMPLE_KW[method])
    frames = [150, 300, 150, 300]
    widths, lens, seeds = [64, 192, 64, 192], [64, 100, 17, 192], [21, 22, 23, 24]
    g = torch.Generator().manual_seed(105)
    texts = [torch.randn(w, cfg.text_dim, generator=g) for w in widths]
    texts = [fill_padding(x[None], [n], "nan_inf")[0].to(dev) for x, n in zip(texts, lens)]
    kw = {}
    if known:
        kp, km = _known(1, 300, cfg.hidden_dim, dev)
        kw = dict(known=[kp[0, :T] for T in frames], known_mask=[km[0, :T] for T in frames])
    out = s.sample_latents_ragged(texts, frames, seeds=seeds, text_lengths=lens, use_graph=use_graph, **kw)
    for i, n in enumerate(lens):
        kwi = {k: [v[i]] for k, v in kw.items()}
        alone = s.sample_latents_ragged([texts[i][:n].contiguous()], [frames[i]], seeds=[seeds[i]], use_graph=use_graph, **kwi)[0]
        assert bool(torch.isfinite(out[i]).all())
        assert rel(out[i], alone) <= SAME_KERNEL_ROW, (i, n, rel(out[i], alone))


def test_ragged_graph_serves_other_lengths(dev):
    """Two jobs with the same (frames, padded width) groups and other text lengths: one capture; the replay equals the eager
    run bitwise; a masked step launches as many kernels as a plain one."""
    cfg, sd, m = model("cross_fused", dev)
    frames, widths, seeds = [150, 150, 300], [64, 64, 64], [31, 32, 33]
    g = torch.Generator().manual_seed(106)
    texts = [torch.randn(w, cfg.text_dim, generator=g).to(dev) for w in widths]
    s = D.DiTTOSampler(m, 3.0, method="ddim", num_steps=6)
    a = s.sample_latents_ragged(texts, frames, seeds=seeds, text_lengths=[64, 10, 33])
    (sig, (ctxs, graphs)), = s._ragged_graphs.items()
    graph = next(iter(graphs.values()))
    b = s.sample_latents_ragged(texts, frames, seeds=seeds, text_lengths=[5, 64, 1])
    assert len(s._ragged_graphs) == 1 and next(iter(next(iter(s._ragged_graphs.values()))[1].values())) is graph
    eager = s.sample_latents_ragged(texts, frames, seeds=seeds, text_lengths=[5, 64, 1], use_graph=False)
    for i in range(3):
        assert torch.equal(b[i], eager[i])
    assert not torch.equal(a[1], b[1])
    plain = D.DiTTOSampler(m, 3.0, method="ddim", num_steps=6)
    plain.sample_latents_ragged(texts, frames, seeds=seeds)
    plain_graph = next(iter(next(iter(plain._ragged_graphs.values()))[1].values()))
    assert graph.launches_per_step == plain_graph.launches_per_step > 0


def test_bad_lengths_are_rejected(dev):
    cfg, sd, m = model("cross_fused", dev)
    x, text, t = inputs(cfg, 2, 150, 64, 107)
    xd, td, tt = x.to(dev), text.to(dev), t.to(dev)
    for bad in ([64], [64, 64, 64], [True, 3], [0, 3], [64, 65], [2.0, 3], "ab"):
        with pytest.raises(D.DittoError):
            m(xd, td, tt, text_lengths=bad)
    s = D.DiTTOSampler(m, 3.0)
    with pytest.raises(D.DittoError):
        s.sample_latents(td, xd, text_lengths=[0, 1])
    with pytest.raises(D.DittoError):
        s.sample_latents_ragged([td[0], td[1, :10]], [150, 150], text_lengths=[64, 11])
    lib = _lib.load()
    ctx = torch.empty(int(lib.ditto_text_context_bytes(m.engine(), 2, 64)), dtype=torch.uint8, device=dev)
    ws = m.workspace(2, 1, 64)
    for bad in ((1, 65), (0, 64), (-3, 1)):
        rc = lib.ditto_text_context_masked(m.engine(), C.c_void_p(td.data_ptr()), 2, 64, (C.c_int64 * 2)(*bad),
                                           C.c_void_p(ctx.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(), None)
        assert rc == -1 and b"[1, S]" in lib.ditto_last_error()
