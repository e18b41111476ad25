"""GPU tests (-m gpu) of csrc/gemm_resid_ln.cu through its C symbol ditto_gemm_resid_ln: the gated MLP's second linear +
bias + fp32 residual (reference: src/components/DiT.py:152-155) and the LayerNorm that follows it (the next block's norm1,
DiT.py:105) in one cluster kernel, against a plain PyTorch fp32 evaluation on the same bf16-rounded operands.  Covers every
supported width (1, 2, 3, 4 column tiles = clusters of 2, 4, 6, 8 CTAs), partial row blocks, more row blocks than
clusters (persistence / barrier parities), and the mode without normalisation (bf16 copy of the residual stream).  Rows with
an offset of up to 4e3 times their spread check the LayerNorm's row statistics alone (reference: the fp64 LayerNorm of the
kernel's own h), per row, next to the two-pass ditto_layernorm on the same rows."""
import ctypes as C

import pytest
import torch

from ditto_tts_b200 import _lib
from oracle import ditto_oracle as O  # rel_l2 only

pytestmark = pytest.mark.gpu
P = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731


def ST():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def run(dev, M, N, K, norm=True, with_u=True, seed=0, h=None, scale=1.0, outputs=False):
    """(rel-L2 of h, of u, h finite) against torch fp32; with outputs=True also (h, u, gamma, beta) as the kernel left them.
    h: the residual stream to start from (default 2 N(0, 1) + 0.5); scale: of the weights and bias (of the increment)."""
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(seed)
    A = torch.randn(M, K, device=dev, generator=g).bfloat16()
    W = (torch.randn(N, K, device=dev, generator=g) * (scale / K ** 0.5)).bfloat16()
    bias = torch.randn(N, device=dev, generator=g) * scale
    h = torch.randn(M, N, device=dev, generator=g) * 2 + 0.5 if h is None else h.to(dev)
    gamma, beta = torch.randn(N, device=dev, generator=g), torch.randn(N, device=dev, generator=g)
    want_h = h + A.float() @ W.float().T + bias
    want_u = torch.nn.functional.layer_norm(want_h, (N,), gamma, beta, 1e-5) if norm else want_h
    perm = torch.tensor([lib.ditto_gemm_resid_ln_weight_row(r) for r in range(N)], device=dev)
    assert sorted(perm.tolist()) == list(range(N))
    Wp = W[perm].contiguous()
    hh = h.clone()
    u = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=dev) if with_u else None
    rc = lib.ditto_gemm_resid_ln(P(A), K, P(Wp), K, P(bias), P(hh), N, P(gamma) if norm else None, P(beta) if norm else None, P(u), N,
                                 M, N, K, ST())
    _lib.check(rc, "ditto_gemm_resid_ln")
    torch.cuda.synchronize()
    eh = O.rel_l2(hh.cpu(), want_h.cpu())
    eu = O.rel_l2(u.float().cpu(), want_u.cpu()) if with_u else 0.0
    if outputs:
        return eh, eu, bool(torch.isfinite(hh).all()), (hh, u, gamma, beta)
    return eh, eu, bool(torch.isfinite(hh).all())


OFFSET_RATIOS = (0.0, 1e2, -1e2, 1e3, -1e3, 4e3, -4e3)   # row offset / row spread
ROW_BAR = 4e-3                                        # per-row rel-L2 of a bf16 output


def offset_rows(M, N, spread, seed):
    """h_r = c_r + spread N(0, 1), c_r / spread drawn per row from OFFSET_RATIOS (all of them appear)."""
    g = torch.Generator().manual_seed(seed)
    ratio = torch.tensor(OFFSET_RATIOS)[torch.arange(M) % len(OFFSET_RATIOS)][torch.randperm(M, generator=g)]
    return ratio[:, None] * spread + spread * torch.randn(M, N, generator=g)


def ln_row_errors(x, y, gamma, beta):
    """Per-row rel-L2 of y (bf16) against the fp64 LayerNorm of x."""
    x64 = x.double().cpu()
    want = torch.nn.functional.layer_norm(x64, (x64.shape[-1],), gamma.double().cpu(), beta.double().cpu(), 1e-5)
    return (y.double().cpu() - want).norm(dim=-1) / want.norm(dim=-1)


@pytest.mark.parametrize("spread", [1.0, 1e-2])
@pytest.mark.parametrize("M,N,K", [(40000, 256, 128), (257, 512, 64), (24000, 768, 256), (513, 1024, 256)])
def test_gemm_resid_ln_row_statistics_under_offset(dev, M, N, K, spread):
    """Row means up to 4e3 x the row spread: the fused LayerNorm must normalise each row of the h it wrote as fp64 would.
    (fp32 E[v^2] - mean^2 loses the whole variance at 4e3 and ~1e-3 of it at 1e2.)  ditto_layernorm, the two-pass kernel,
    takes the same rows to the same bar."""
    h = offset_rows(M, N, spread, seed=M + N)
    eh, _, finite, (hh, u, gamma, beta) = run(dev, M, N, K, h=h, scale=spread, outputs=True)   # increment ~ spread
    rows = ln_row_errors(hh, u.float(), gamma, beta)
    assert finite and eh <= 1e-4, eh
    assert float(rows.max()) <= ROW_BAR, (float(rows.max()), int(rows.argmax()), float(hh[int(rows.argmax())].mean()))
    lib = _lib.load()
    y = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=dev)
    _lib.check(lib.ditto_layernorm(P(hh), P(gamma), P(beta), P(y), 1, M, N, ST()), "ditto_layernorm")
    torch.cuda.synchronize()
    rows2 = ln_row_errors(hh, y.float(), gamma, beta)
    assert float(rows2.max()) <= ROW_BAR, float(rows2.max())


@pytest.mark.parametrize("M,N,K", [(1000, 768, 3072), (24000, 768, 3072), (100, 256, 512), (257, 512, 64), (513, 1024, 256),
                                   (1, 768, 768), (40000, 256, 128)])
def test_gemm_resid_ln_vs_torch(dev, M, N, K):
    eh, eu, finite = run(dev, M, N, K)
    assert finite and eh <= 2e-6 * 50 and eu <= 4e-3, (eh, eu)


@pytest.mark.parametrize("M,N,K", [(1000, 768, 3072), (300, 256, 512)])
def test_gemm_resid_without_layernorm(dev, M, N, K):
    eh, eu, finite = run(dev, M, N, K, norm=False)
    assert finite and eh <= 1e-4 and eu <= 4e-3, (eh, eu)
    eh, _, finite = run(dev, M, N, K, norm=False, with_u=False)
    assert finite and eh <= 1e-4


def test_gemm_resid_ln_rejects_bad_arguments(dev):
    lib = _lib.load()
    A = torch.zeros(8, 64, dtype=torch.bfloat16, device=dev)
    W = torch.zeros(256, 64, dtype=torch.bfloat16, device=dev)
    b = torch.zeros(256, device=dev)
    h = torch.zeros(8, 256, device=dev)
    u = torch.zeros(8, 256, dtype=torch.bfloat16, device=dev)
    assert lib.ditto_gemm_resid_ln(None, 64, P(W), 64, P(b), P(h), 256, None, None, None, 256, 8, 256, 64, ST()) == -1
    assert lib.ditto_gemm_resid_ln(P(A), 64, P(W), 64, P(b), P(h), 256, P(b), None, P(u), 256, 8, 256, 64, ST()) == -1   # gamma without beta
    assert lib.ditto_gemm_resid_ln(P(A), 64, P(W), 64, P(b), P(h), 256, None, None, None, 256, 8, 320, 64, ST()) != 0    # unsupported width
