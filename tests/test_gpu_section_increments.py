"""GPU tests (-m gpu) of the DiT block sections by their increment: ``blk.section(name, x, text) - x`` and ``blk(x, text) - x``
against the fp64 increment of the oracle (oracle/section_ref.py: cases, inputs, bars).

The sum ``x + f(x)`` that the block returns is ~90 % residual, so a bar on it lets a self-attention that skips RoPE or returns
the mean of V pass; the increment does not.  The cases cover the kernels each section can take on the bf16 path -- the QKV +
RoPE and GEGLU epilogues, flash_attn768 / flash_attn768q, flash_attn_d64, cross_fused, flash_attn768q<CROSS> (including its
online-softmax rescale), the cluster scores + softmax kernel with row_lsum -- with default and sharpened (peaked softmax)
weights, and again under the developer switches that select another kernel for the same section.  Each run also checks that
the kernel class it was meant to exercise actually ran.  tests/test_section_sensitivity.py guards the bars on the CPU."""
import functools

import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from oracle import section_ref as R  # checker only

pytestmark = pytest.mark.gpu

F768, SELF_PV, FLASH64 = "tc_gemm.flash768_ln", "tc_gemm.self_pv", "tc_gemm.flash_attn"
XFUSED, XFLASH, XPV = "tc_gemm.cross_fused_ln", "tc_gemm.cross_flash_ln", "tc_gemm.cross_pv"


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@functools.lru_cache(maxsize=None)
def reference(name):
    """(cfg, sd, x, text, fp64 increments) of a case, computed once per session."""
    case = R.CASE[name]
    cfg, sd, x, text = R.case_inputs(case)
    return cfg, sd, x, text, R.increments(case, sd, x, text)


def build_model(cfg, sd, precision, dev):
    m = D.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=cfg.num_heads, time_dim=cfg.time_dim,
                text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps, precision=precision)
    m.load_state_dict(sd, strict=True)
    return m.to(dev)


def expected_kernels(case, opts):
    """section -> (kernel classes that must run, classes that must not) on the bf16 path under the debug options ``opts``,
    following the engine's selection (engine.cu: engine_create, forward_impl)."""
    on = lambda k: bool(opts.get(k, 0))  # noqa: E731
    one768 = case.hidden == 768 and case.heads == 1
    flash768 = one768 and not (on("no_flash768") or on("no_pv_perm4") or on("rope_generic") or on("defer_ln2"))
    folded = case.heads * ((case.S + 7) // 8 * 8) * 2 <= case.hidden
    fused_cross = one768 and folded and not on("no_fused_cross")
    if one768:
        self_k = ((F768,), ()) if flash768 else ((SELF_PV,), (F768,))
    else:
        self_k = ((SELF_PV,), (FLASH64,)) if on("no_flash") else ((FLASH64,), ())
    if fused_cross and case.S <= 64:
        cross_k = ((XFUSED,), ())
    elif fused_cross and case.S <= 256 and flash768 and not (on("no_cross_flash") or on("no_fc2_ln")):
        cross_k = ((XFLASH,), ())
    else:
        cross_k = ((XPV,), (XFUSED, XFLASH))
    return {"self": self_k, "cross": cross_k}


def run_and_check(case, precision, dev, opts=None):
    opts = opts or {}
    cfg, sd, x, text, want = reference(case.name)
    got, ran = {}, {}
    for k, v in opts.items():
        _lib.debug_option(k, v)
    try:
        m = build_model(cfg, sd, precision, dev)       # kept alive: a block whose model is gone runs on a bf16 engine of its own
        blk = m.blocks[R.LAYER]
        xd, td = x.to(dev), text.to(dev)
        for s in case.sections:
            _lib.profile_start()
            try:
                out = blk(xd, td) if s == "block" else blk.section(s, xd, td)
            finally:
                prof = _lib.profile_stop()
            got[s], ran[s] = out.cpu(), set(prof)
    finally:
        _lib.debug_option("reset", 0)
    report, bad = [], []
    for s in case.sections:
        finite = bool(torch.isfinite(got[s]).all())
        e, row = R.errors(got[s].double() - x.double(), want[s])
        b, rb = R.bar(case, precision, s), R.row_bar(case, precision, s)
        report.append(f"{s}={e:.2e}/{row:.2e} (bar {b:.0e}{'' if rb is None else f'/{rb:.1e}'})")
        if not finite or e > b or (rb is not None and row > rb):
            bad.append(s)
    opt_s = "+".join(f"{k}={v}" for k, v in opts.items()) or "default"
    print(f"[section-increment] {case.name} {precision} {opt_s}: " + "  ".join(report))
    assert not bad, (case.name, precision, opts, bad, report)
    if precision == "bf16":
        for s, (must, must_not) in expected_kernels(case, opts).items():
            if s in ran:
                assert set(must) <= ran[s] and not set(must_not) & ran[s], (case.name, s, opts, sorted(ran[s]))


@pytest.mark.parametrize("name", [c.name for c in R.CASES])
def test_section_increments_bf16(dev, name):
    run_and_check(R.CASE[name], "bf16", dev)


@pytest.mark.parametrize("name", [c.name for c in R.CASES if c.fp32])
def test_section_increments_fp32(dev, name):
    run_and_check(R.CASE[name], "fp32", dev)


ONE_HEAD_T = ("t1", "t129", "t257", "t750_sharp", "t2250")
SWITCH_RUNS = [
    ({"flash768_quad": 1}, ONE_HEAD_T + ("load",)),            # two-CTA flash_attn768 at every length
    ({"flash768_quad": 2}, ONE_HEAD_T + ("load",)),            # four-CTA flash_attn768q at every length
    ({"no_flash768": 1}, ONE_HEAD_T),
    ({"no_flash": 1}, ("h12_t130_s9", "h12_t257_s100_sharp", "h12_t750_s100", "h256_t300", "h128_t77")),
    ({"no_fused_cross": 1}, ("s1", "s64", "s64_sharp", "s65", "s129_sharp", "s256", "s200_loud_sharp")),
    ({"no_cross_flash": 1}, ("s65", "s128", "s129_sharp", "s256", "s200_loud", "s200_loud_sharp")),
    ({"rope_generic": 1, "glu_generic": 1}, ("t129", "t750_sharp", "s129", "h12_t257_s9", "h256_t300")),
    ({"no_pv_perm4": 1}, ("t129", "t750_sharp", "s129")),
    ({"no_fc2_ln": 1}, ("t257", "s65", "s129_sharp", "s512", "s512_sharp")),
    ({"defer_ln2": 1}, ("t129", "t750_sharp", "s1", "s64", "s64_sharp")),
]


@pytest.mark.parametrize("opts,name", [(o, n) for o, names in SWITCH_RUNS for n in names],
                         ids=[f"{'+'.join(f'{k}={v}' for k, v in o.items())}-{n}" for o, names in SWITCH_RUNS for n in names])
def test_section_increments_under_switch(dev, opts, name):
    run_and_check(R.CASE[name], "bf16", dev, opts)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["t257", "s129", "h12_t130_s9", "h256_t77"])
def test_sections_chain_to_the_whole_block(dev, name, precision):
    """self -> cross -> mlp through the section entry points == the whole block (ditto_dit_block); a bad name is refused."""
    cfg, sd, x, text, _ = reference(name)
    m = build_model(cfg, sd, precision, dev)
    blk = m.blocks[R.LAYER]
    xd, td = x.to(dev), text.to(dev)
    chained = blk.section("mlp", blk.section("cross", blk.section("self", xd, td), td), td)
    whole = blk(xd, td)
    assert R.errors(chained, whole)[0] <= (1e-5 if precision == "fp32" else 6e-3)
    with pytest.raises(D.DittoError):
        blk.section("attn", xd, td)
