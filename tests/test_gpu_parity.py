"""Parity tests proper (-m gpu): the CUDA path, called through the C-ABI, against
  (a) golden outputs of the UNMODIFIED reference (tests/golden/*.npz, minted by make_golden.py), and
  (b) the CPU oracle on the same seeded inputs.
Bars (BASELINE.json north_star): rel-L2 <= 1e-4 for the fp32 path, <= 2e-2 for the bf16 path, per-step
denoiser output and final latent.  /root/reference is never read here."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from oracle import ditto_oracle as O

pytestmark = pytest.mark.gpu
BAR = {"fp32": 1e-4, "bf16": 2e-2}
P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731


def ST():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def build_model(cfg, sd, precision, dev, fused_rope=True, fold_cross=None, defer_ln=False):
    """fused_rope=False runs the plain composition (separate RoPE / LayerNorm / projection kernels);
    fused_rope="defer_ln" adds the LayerNorm folding (DITTO_F_DEFER_LN) to the default fusions."""
    if fused_rope == "defer_ln":
        fused_rope, defer_ln = True, True
    fold_cross = fused_rope if fold_cross is None else fold_cross
    m = D.DiTTO(hidden_dim=cfg.hidden_dim, num_layers=cfg.num_layers, num_heads=cfg.num_heads, time_dim=cfg.time_dim,
                text_dim=cfg.text_dim, diffusion_steps=cfg.diffusion_steps, precision=precision, fused_rope=fused_rope,
                fold_cross=fold_cross, defer_ln=defer_ln)
    m.load_state_dict(sd, strict=True)
    return m.to(dev)


def rel(a, b):
    return O.rel_l2(a.float().cpu(), b.float().cpu())


# ------------------------------------------------------------------------------------------ operators
@pytest.mark.parametrize("rows,H", [(37, 768), (5, 64), (1000, 1024), (1, 8)])
def test_layernorm(dev, rows, H):
    lib = _lib.load()
    g = torch.Generator().manual_seed(0)
    x = torch.randn(rows, H, generator=g) * 3 + 1
    ga, be = torch.randn(H, generator=g), torch.randn(H, generator=g)
    ref = torch.nn.functional.layer_norm(x, (H,), ga, be, 1e-5)
    xd, gd, bd = x.to(dev), ga.to(dev), be.to(dev)
    y = torch.empty_like(xd)
    _lib.check(lib.ditto_layernorm(P(xd), P(gd), P(bd), P(y), 0, rows, H, ST()))
    assert rel(y, ref) <= 1e-6
    yb = torch.empty(rows, H, dtype=torch.bfloat16, device=dev)
    _lib.check(lib.ditto_layernorm(P(xd), P(gd), P(bd), P(yb), 1, rows, H, ST()))
    assert rel(yb, ref) <= 4e-3      # bf16 rounding of the output only
    _lib.check(lib.ditto_layernorm(P(xd), None, None, P(y), 0, rows, H, ST()))
    assert rel(y, torch.nn.functional.layer_norm(x, (H,))) <= 1e-6


def test_layernorm_rejects_unsupported_width(dev):
    lib = _lib.load()
    x = torch.zeros(2, 1030, device=dev)
    assert lib.ditto_layernorm(P(x), None, None, P(x), 0, 2, 1030, ST()) == -2
    assert lib.ditto_layernorm(P(x), None, None, P(x), 0, 0, 1024, ST()) == 0   # empty input is a no-op


@pytest.mark.parametrize("M,N,K,batch,nk", [(130, 70, 33, 1, 1), (257, 129, 768, 2, 1), (64, 300, 50, 3, 0),
                                            (750, 768, 750, 2, 0), (1, 1, 1, 1, 1)])
def test_gemm_f32(dev, M, N, K, batch, nk):
    lib = _lib.load()
    g = torch.Generator().manual_seed(1)
    A = torch.randn(batch, M, K, generator=g)
    B = torch.randn(batch, N, K, generator=g) if nk else torch.randn(batch, K, N, generator=g)
    bias, R = torch.randn(N, generator=g), torch.randn(batch, M, N, generator=g)
    ref = 0.5 * (A.double() @ (B.double().transpose(1, 2) if nk else B.double())) + bias + R
    Ad, Bd, bd, Rd = A.to(dev), B.to(dev), bias.to(dev), R.to(dev)
    Cd = torch.empty(batch, M, N, device=dev)
    _lib.check(lib.ditto_gemm_f32(P(Ad), K, M * K, P(Bd), K if nk else N, N * K, nk, P(Cd), N, M * N, P(bd), P(Rd), 0.5,
                                  M, N, K, batch, ST()))
    assert rel(Cd, ref) <= 2e-6


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (1, 8, 8), (300, 200, 136), (300, 201, 136), (1000, 768, 768),
                                   (750, 750, 768), (4096, 768, 3072), (24000, 2304, 768)])
def test_gemm_bf16_tcgen05(dev, M, N, K):
    """tcgen05 GEMM == fp32 matmul of the same bf16 operands up to accumulation order (fp32 accumulators in TMEM).
    Covers every STORE-epilogue variant: fp32 / bf16 output, with / without residual, residual in place, odd N."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(2)
    A = torch.randn(M, K, generator=g).bfloat16().to(dev)
    W = (torch.randn(N, K, generator=g) / K ** 0.5).bfloat16().to(dev)
    bias = torch.randn(N, generator=g).to(dev)
    ldc = (N + 7) // 8 * 8
    R = torch.randn(M, ldc, generator=g).to(dev)
    R[:, N:] = 0
    base = 0.25 * (A.float() @ W.float().T) + bias
    for out_bf16 in (0, 1):
        for use_resid in (True, False):
            ref = base + R[:, :N] if use_resid else base
            Cd = torch.zeros(M, ldc, dtype=torch.bfloat16 if out_bf16 else torch.float32, device=dev)
            _lib.check(lib.ditto_gemm_bf16(P(A), K, P(W), K, P(Cd), ldc, out_bf16, P(bias), P(R) if use_resid else None, ldc,
                                           0.25, M, N, K, ST()))
            assert rel(Cd[:, :N], ref) <= (4e-3 if out_bf16 else 2e-5), (out_bf16, use_resid)
            if ldc > N:
                assert float(Cd[:, N:].abs().max()) == 0.0   # padding columns untouched
    # residual updated in place (how the engine keeps the fp32 residual stream h)
    Cd = R.clone()
    _lib.check(lib.ditto_gemm_bf16(P(A), K, P(W), K, P(Cd), ldc, 0, P(bias), P(Cd), ldc, 0.25, M, N, K, ST()))
    assert rel(Cd[:, :N], base + R[:, :N]) <= 2e-5
    if ldc > N:
        assert float(Cd[:, N:].abs().max()) == 0.0


def test_gemm_bf16_rejects_misaligned(dev):
    lib = _lib.load()
    A = torch.zeros(16, 12, dtype=torch.bfloat16, device=dev)
    Cd = torch.zeros(16, 16, device=dev)
    assert lib.ditto_gemm_bf16(P(A), 12, P(A), 12, P(Cd), 16, 0, None, None, 0, 1.0, 16, 16, 12, ST()) == -2


@pytest.mark.parametrize("guided", [True, False])
def test_cfg_ddpm_update_and_q_sample(dev, guided):
    lib = _lib.load()
    cfg = O.OracleConfig(64, 1, 2, 32, 64, 50)
    sd = O.make_state_dict(cfg, 0)
    m = build_model(cfg, sd, "fp32", dev)
    D.DiTTOSampler(m)
    g = torch.Generator().manual_seed(3)
    B, T, H, w = 3, 10, 64, 3.0
    ec, eu, x, z = (torch.randn(B, T, H, generator=g) for _ in range(4))
    t = torch.tensor([49, 0, 17])
    betas, alphas, acp = O.sampler_tables(50)
    ref = O.p_sample_update(x, eu + w * (ec - eu) if guided else ec, z, t, betas, alphas, acp)
    ecd, eud, xd, zd, td = ec.to(dev), eu.to(dev), x.to(dev), z.to(dev), t.to(dev)
    out = torch.empty(B, T, H, device=dev)
    _lib.check(lib.ditto_cfg_ddpm_update(m.engine(), P(ecd), P(eud) if guided else None, P(xd), P(zd), P(td), w, P(out), B,
                                         T * H, ST()))
    assert rel(out, ref) <= 1e-6
    assert torch.equal(out[1].cpu(), ref[1]) or rel(out[1], ref[1]) <= 1e-6     # t = 0: no noise term
    # in place (x_out aliases x) and empty batch
    _lib.check(lib.ditto_cfg_ddpm_update(m.engine(), P(ecd), P(eud) if guided else None, P(xd), P(zd), P(td), w, P(xd), B,
                                         T * H, ST()))
    assert rel(xd, ref) <= 1e-6
    assert lib.ditto_cfg_ddpm_update(m.engine(), P(ecd), None, P(xd), None, P(td), w, P(out), 0, T * H, ST()) == 0
    qs = m.q_sample(x.to(dev), t.to(dev), z.to(dev))
    assert rel(qs, O.q_sample(sd, x, t, z)) <= 1e-6


# ------------------------------------------------------------------------------------------ forward
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_tiny_forward_vs_reference_golden(dev, golden, precision):
    g = golden("tiny_full.npz")
    cfg = O.OracleConfig(*[int(v) for v in g["cfg"]])
    sd = {k[4:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd::")}
    m = build_model(cfg, sd, precision, dev)
    out = m(torch.from_numpy(g["x"]).to(dev), torch.from_numpy(g["text"]).to(dev), torch.from_numpy(g["t"]).to(dev))
    assert rel(out, torch.from_numpy(g["out"])) <= BAR[precision]


@pytest.mark.parametrize("precision,fused", [("fp32", True), ("bf16", True), ("bf16", "defer_ln"), ("bf16", False)])
@pytest.mark.parametrize("name", ["c1_default", "ctor_default", "ragged"])
def test_full_size_forward_vs_reference_golden(dev, golden, name, precision, fused):
    """C1 (B=1, T=750, S=64, repo-default 5 layers x 1 head of 768), the constructor-default model
    (12 layers x 12 heads of 64) and a ragged shape (T=173, S=19, per-sequence t incl. t=0 and t=steps-1)."""
    f = golden("full_size.npz")
    meta = [int(v) for v in f[f"{name}::meta"]]
    cfg = O.OracleConfig(*meta[:6])
    wseed, iseed, B, T, S, stride = meta[6:]
    sd = O.make_state_dict(cfg, wseed)
    x, text, _ = O.make_inputs(B, T, S, cfg, iseed)
    t = torch.from_numpy(f[f"{name}::t"])
    m = build_model(cfg, sd, precision, dev, fused)
    out = m(x.to(dev), text.to(dev), t.to(dev))
    assert rel(out[:, ::stride], torch.from_numpy(f[f"{name}::out_sub"])) <= BAR[precision]
    assert abs(float(out.double().norm()) / float(f[f"{name}::out_norm"][0]) - 1) <= BAR[precision]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_forward_vs_oracle_odd_shapes(dev, precision):
    """Edge shapes against the CPU oracle: T not a multiple of any tile, S = 1, single frame, shared x (CFG layout)."""
    cfg = O.OracleConfig(768, 2, 1, 256, 768, 20)
    sd = O.make_state_dict(cfg, 11)
    m = build_model(cfg, sd, precision, dev)
    for (B, T, S) in ((1, 1, 1), (3, 129, 5), (2, 257, 70)):
        x, text, _ = O.make_inputs(B, T, S, cfg, 12)
        t = torch.arange(B) % cfg.diffusion_steps
        ref = O.ditto_forward(sd, cfg, x, text, t)
        out = m(x.to(dev), text.to(dev), t.to(dev))
        assert rel(out, ref) <= BAR[precision], (B, T, S)
    # shared-x batch: n_seq = 2 n_x, second half sees zero text (the CFG layout)
    B, T, S = 2, 64, 9
    x, text, _ = O.make_inputs(B, T, S, cfg, 13)
    t = torch.tensor([3, 3, 3, 3])
    both = torch.cat([text, torch.zeros_like(text)])
    ctx = m.text_context(both.to(dev), T_hint=T)
    out = m.forward_with_context(x.to(dev), ctx, t.to(dev), 4, S)
    ref = O.ditto_forward(sd, cfg, torch.cat([x, x]), both, t)
    assert rel(out, ref) <= BAR[precision]


@pytest.mark.parametrize("fused", [True, "defer_ln"])
def test_layernorm_folding_with_offset_rows(dev, fused):
    """Deferred LayerNorm consumes bf16(h) and per-row (sum, sum of squares) instead of LN(h): rows whose mean is several
    standard deviations away from zero (AdaLN shift biased by +4) and a multi-head model (per-head statistics parts,
    materialised LN2) must still meet the bf16 bar."""
    for heads, (B, T, S) in ((1, (2, 300, 33)), (4, (2, 131, 40))):
        cfg = O.OracleConfig(256, 2, heads, 64, 256, 20)
        sd = O.make_state_dict(cfg, 41)
        sd["ada_ln.time_mlp.1.bias"][cfg.hidden_dim:] += 4.0
        x, text, _ = O.make_inputs(B, T, S, cfg, 42)
        t = torch.tensor([0, 19])
        ref = O.ditto_forward(sd, cfg, x, text, t)
        out = build_model(cfg, sd, "bf16", dev, fused)(x.to(dev), text.to(dev), t.to(dev))
        assert rel(out, ref) <= BAR["bf16"], (heads, rel(out, ref))


def test_long_sequence_bf16_vs_oracle(dev):
    """30 s utterance (T = 2250, beyond the reference's data cap but valid for the module), attention-dominated."""
    cfg = O.OracleConfig(768, 1, 1, 256, 768, 20)
    sd = O.make_state_dict(cfg, 21)
    x, text, _ = O.make_inputs(1, 2250, 192, cfg, 22)
    t = torch.tensor([4])
    ref = O.ditto_forward(sd, cfg, x, text, t)
    out = build_model(cfg, sd, "bf16", dev)(x.to(dev), text.to(dev), t.to(dev))
    assert rel(out, ref) <= 2e-2


# ------------------------------------------------------------------------------------------ sampler
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_reference_sampler_loop_tiny(dev, golden, precision):
    """The reference's own __p_sample loop (no guidance, 8 steps), noise replayed."""
    g = golden("tiny_full.npz")
    cfg = O.OracleConfig(*[int(v) for v in g["cfg"]])
    sd = {k[4:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd::")}
    s = D.DiTTOSampler(build_model(cfg, sd, precision, dev))
    out = s.sample_latents(torch.from_numpy(g["text"]).to(dev), x_init=torch.from_numpy(g["x"]).to(dev),
                           noise=torch.from_numpy(g["ref_noise"]).to(dev))
    assert rel(out, torch.from_numpy(g["sampled"])) <= BAR[precision]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_cfg_50_steps_vs_reference_trajectory(dev, golden, precision):
    """Full 50-step CFG sampling (w = 3, uncond = zero text) on the default model, B=2, T=96: first and last
    per-step eps_hat and the final latent (every `stride`-th frame, plus the norms of the full tensors) against the
    trajectory computed with the reference forward."""
    c = golden("cfg_traj.npz")
    B, T, S, iseed, wseed, steps = [int(v) for v in c["meta"]]
    stride = int(c["stride"][0])
    cfg = O.OracleConfig(768, 5, 1, 256, 768, steps)
    sd = O.make_state_dict(cfg, wseed)
    x, text, noise = O.make_inputs(B, T, S, cfg, iseed, steps_noise=steps)
    s = D.DiTTOSampler(build_model(cfg, sd, precision, dev), guidance_scale=float(c["w"][0]))
    rec = []
    out = s.sample_latents(text.to(dev), x_init=x.to(dev), noise=noise.to(dev), record=rec)
    assert len(rec) == steps
    assert rel(rec[0][:, ::stride], torch.from_numpy(c["eps_first"])) <= BAR[precision]
    assert rel(rec[-1][:, ::stride], torch.from_numpy(c["eps_last"])) <= BAR[precision]
    assert rel(out[:, ::stride], torch.from_numpy(c["final"])) <= BAR[precision]
    assert abs(float(out.double().norm()) / float(c["final_norm"][0]) - 1.0) <= BAR[precision]
    norms = np.array([float(e.double().norm()) for e in rec])
    assert np.allclose(norms, c["eps_norms"], rtol=BAR[precision])


def test_full_size_batch_properties_bf16(dev):
    """BASELINE config C2 at full size (B=16, T=750, S=64), size-independent properties instead of a CPU run:
    (i) batch independence: utterance i of the batch == the same utterance run alone;
    (ii) a CFG step with w = 1 equals the unguided step;  (iii) outputs finite."""
    cfg = O.OracleConfig(768, 5, 1, 256, 768, 50)
    sd = O.make_state_dict(cfg, 0)
    m = build_model(cfg, sd, "bf16", dev)
    s = D.DiTTOSampler(m)
    x, text, noise = O.make_inputs(16, 750, 64, cfg, 31, steps_noise=1)
    xd, td, zd = x.to(dev), text.to(dev), noise[0].to(dev)
    t = torch.full((16,), 42, dtype=torch.long, device=dev)
    full = s.p_sample(xd, t, td, noise=zd, guidance_scale=3.0)
    assert bool(torch.isfinite(full).all())
    one = s.p_sample(xd[5:6], t[:1], td[5:6], noise=zd[5:6], guidance_scale=3.0)
    assert rel(full[5:6], one) <= 1e-5                      # same kernels, same per-row arithmetic
    unguided = s.p_sample(xd, t, td, noise=zd, guidance_scale=None)
    w1 = s.p_sample(xd, t, td, noise=zd, guidance_scale=1.0)
    assert rel(w1, unguided) <= 1e-5
    assert _lib.launch_count() > 0


# ------------------------------------------------------------------------------------------ fused cross-attention block
@pytest.mark.parametrize("B,T,S", [(2, 750, 64), (3, 130, 5), (1, 1, 1), (2, 257, 33), (1, 128, 64)])
def test_fused_cross_attention_block(dev, B, T, S):
    """cross_fused.cu (scores + softmax + P.V + residual + norm3 in one kernel) against the oracle and against the
    separate-kernel composition (debug option no_fused_cross), default single-head model, bf16 path."""
    cfg = O.OracleConfig(768, 2, 1, 256, 768, 50)
    sd = O.make_state_dict(cfg, 21)
    x, text, _ = O.make_inputs(B, T, S, cfg, 22)
    t = torch.arange(B) * 7 + 3
    want = O.ditto_forward(sd, cfg, x, text, t)
    outs = {}
    for fused in (True, False):
        _lib.debug_option("no_fused_cross", 0 if fused else 1)
        try:
            m = build_model(cfg, sd, "bf16", dev)
            _lib.profile_start()
            outs[fused] = m(x.to(dev), text.to(dev), t.to(dev))
            prof = _lib.profile_stop()
        finally:
            _lib.debug_option("reset", 0)
        assert ("tc_gemm.cross_fused_ln" in prof) == fused, sorted(prof)
        assert ("tc_gemm.cross_pv" in prof) == (not fused)
        assert rel(outs[fused], want) <= BAR["bf16"]
    assert rel(outs[True], outs[False]) <= 6e-3     # same operands, different rounding points of P / LN statistics


@pytest.mark.parametrize("B,T,S", [(2, 750, 65), (1, 300, 100), (2, 257, 128), (1, 130, 129), (1, 2250, 192), (2, 90, 256)])
def test_flash_cross_attention_block(dev, B, T, S):
    """flash_attn768q<CROSS> (64 < S <= 256 text tokens: scores, online softmax over up to two key tiles, P (V Wo^T), + bo +
    residual + norm3 in one cluster kernel) against the oracle and against the three-kernel composition (no_cross_flash)."""
    cfg = O.OracleConfig(768, 2, 1, 256, 768, 50)
    sd = O.make_state_dict(cfg, 23)
    x, text, _ = O.make_inputs(B, T, S, cfg, 24)
    t = torch.arange(B) * 11 + 5
    want = O.ditto_forward(sd, cfg, x, text, t)
    outs = {}
    for fused in (True, False):
        _lib.debug_option("no_cross_flash", 0 if fused else 1)
        try:
            m = build_model(cfg, sd, "bf16", dev)
            _lib.profile_start()
            outs[fused] = m(x.to(dev), text.to(dev), t.to(dev))
            prof = _lib.profile_stop()
        finally:
            _lib.debug_option("reset", 0)
        assert ("tc_gemm.cross_flash_ln" in prof) == fused, sorted(prof)
        assert ("tc_gemm.cross_pv" in prof) == (not fused)
        assert rel(outs[fused], want) <= BAR["bf16"], rel(outs[fused], want)
    assert rel(outs[True], outs[False]) <= 6e-3


@pytest.mark.parametrize("B,T,S,switch,cls", [(48, 750, 64, "no_fused_cross", "tc_gemm.cross_fused_ln"),
                                              (24, 750, 100, "no_cross_flash", "tc_gemm.cross_flash_ln"),
                                              (40, 750, 64, "no_flash768", "tc_gemm.flash768_ln")])
def test_fused_blocks_under_load_match_their_compositions(dev, B, T, S, switch, cls):
    """The one-kernel blocks with several tiles / items per CTA or cluster (the shapes above give each CTA a single one, where a
    hand-over hazard between consecutive tiles cannot show) against the separate-kernel composition of the same arithmetic."""
    cfg = O.OracleConfig(768, 2, 1, 256, 768, 50)
    sd = O.make_state_dict(cfg, 25)
    x, text, _ = O.make_inputs(B, T, S, cfg, 26)
    t = (torch.arange(B) * 5 + 1) % 50
    outs = {}
    for fused in (True, False):
        _lib.debug_option(switch, 0 if fused else 1)
        try:
            m = build_model(cfg, sd, "bf16", dev)
            _lib.profile_start()
            outs[fused] = m(x.to(dev), text.to(dev), t.to(dev))
            prof = _lib.profile_stop()
        finally:
            _lib.debug_option("reset", 0)
        assert (cls in prof) == fused, sorted(prof)
    assert torch.isfinite(outs[True]).all()
    assert rel(outs[True], outs[False]) <= 6e-3, rel(outs[True], outs[False])


@pytest.mark.parametrize("env", [{"xf_rows": 88}, {"defer_ln2": 1}, {"rope_generic": 1, "glu_generic": 1}, {"no_pv_perm4": 1},
                                 {"no_flash768": 1}, {"no_fused_ln": 1}, {"no_fc2_ln": 1}, {"flash768_quad": 1}, {"no_cross_flash": 1}],
                         ids=lambda e: "+".join(f"{k}={v}" for k, v in e.items()))
def test_kernel_variants_behind_switches(dev, env):
    """Every developer switch of DESIGN.md section 9 selects a different kernel / weight packing for the same arithmetic: each
    must stay within the bf16 bar of the oracle and within rounding of the default build (C2 width, ragged T, S = 40)."""
    cfg = O.OracleConfig(768, 2, 1, 256, 768, 50)
    sd = O.make_state_dict(cfg, 41)
    x, text, _ = O.make_inputs(2, 300, 40, cfg, 42)
    t = torch.tensor([49, 0])
    want = O.ditto_forward(sd, cfg, x, text, t)
    base = build_model(cfg, sd, "bf16", dev)(x.to(dev), text.to(dev), t.to(dev))
    for k, v in env.items():
        _lib.debug_option(k, v)
    try:
        got = build_model(cfg, sd, "bf16", dev)(x.to(dev), text.to(dev), t.to(dev))
    finally:
        _lib.debug_option("reset", 0)
    assert rel(got, want) <= BAR["bf16"]
    assert rel(base, want) <= BAR["bf16"]
    assert rel(got, base) <= 8e-3


@pytest.mark.parametrize("B,T,S,hidden,heads", [(2, 750, 20, 256, 4), (3, 130, 7, 128, 2), (1, 1, 3, 64, 1), (2, 257, 9, 768, 12),
                                                (1, 128, 5, 192, 3)])
def test_flash_attention_d64(dev, B, T, S, hidden, heads):
    """flash_attn.cu (head_dim 64: two-pass attention, scores and probabilities never in HBM) against the oracle and
    against the GEMM formulation (debug option no_flash): multi-head models, ragged T, partial key tiles."""
    cfg = O.OracleConfig(hidden, 2, heads, 64, hidden, 20)
    sd = O.make_state_dict(cfg, 51)
    x, text, _ = O.make_inputs(B, T, S, cfg, 52)
    t = (torch.arange(B) * 5 + 1) % 20
    want = O.ditto_forward(sd, cfg, x, text, t)
    outs = {}
    for flash in (True, False):
        _lib.debug_option("no_flash", 0 if flash else 1)
        try:
            m = build_model(cfg, sd, "bf16", dev)
            _lib.profile_start()
            outs[flash] = m(x.to(dev), text.to(dev), t.to(dev))
            prof = _lib.profile_stop()
        finally:
            _lib.debug_option("reset", 0)
        assert ("tc_gemm.flash_attn" in prof) == flash, sorted(prof)
        assert ("tc_gemm.self_pv" in prof) == (not flash)
        assert bool(torch.isfinite(outs[flash]).all())
        assert rel(outs[flash], want) <= BAR["bf16"]
    assert rel(outs[True], outs[False]) <= 8e-3
