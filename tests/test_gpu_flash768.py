"""GPU tests (-m gpu) of flash_attn768.cu / flash_attn768q.cu through its C symbol ditto_attn_self768: self-attention of ONE head of 768
(reference: src/components/DiT.py:117-139, repo-default config) + residual + norm2 in one cluster kernel, against a plain
PyTorch fp32 evaluation of the same formulas on the same bf16-rounded operands.  Covers partial query / key tiles, long
sequences, and the online-softmax rescale path (forced, and provoked by keys whose scores grow along the sequence)."""
import ctypes as C
import math

import pytest
import torch

from ditto_tts_b200 import _lib
from oracle import ditto_oracle as O  # rel_l2 only

pytestmark = pytest.mark.gpu
P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
H = 768


def ST():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(autouse=True, params=["pair", "quad"])
def kernel_variant(request):
    """Every test runs on both kernels: flash_attn768_kernel (two-CTA cluster, 128 query rows) and flash_attn768q_kernel (four-CTA
    cluster of two cta_group::2 pairs, 256 query rows) -- the launcher otherwise picks by sequence length."""
    _lib.debug_option("flash768_quad", 1 if request.param == "pair" else 2)
    yield request.param
    _lib.debug_option("flash768_quad", 0)


def v_storage_order():
    """position l of every 64-column block -> logical column (include/ditto_b200.h, ditto_attn_self768)."""
    idx = torch.empty(H, dtype=torch.long)
    for b in range(H // 64):
        for kb in range(8):
            for q in range(4):
                for e in range(2):
                    idx[64 * b + 8 * kb + 2 * q + e] = 64 * b + 16 * (kb // 2) + 4 * q + 2 * (kb % 2) + e
    return idx


def reference(q, k, v, h, gamma, beta, alpha):
    s = torch.einsum("ntd,nsd->nts", q.float(), k.float()) * alpha
    o = torch.softmax(s, dim=-1) @ v.float()
    hn = h + o
    return hn, torch.nn.functional.layer_norm(hn, (H,), gamma, beta, 1e-5), o


def run(dev, n, T, flags=0, key_scale=None, seed=0, with_ln=True):
    g = torch.Generator(device=dev).manual_seed(seed)
    q = torch.randn(n, T, H, device=dev, generator=g).bfloat16()
    k = torch.randn(n, T, H, device=dev, generator=g)
    if key_scale is not None:
        k = k * key_scale(torch.arange(T, device=dev)).view(1, T, 1)
    k = k.bfloat16()
    v = torch.randn(n, T, H, device=dev, generator=g).bfloat16()
    h = torch.randn(n, T, H, device=dev, generator=g) * 2
    gamma, beta = torch.randn(H, device=dev, generator=g), torch.randn(H, device=dev, generator=g)
    alpha = 1.0 / math.sqrt(H)
    want_h, want_u, want_o = reference(q, k, v, h, gamma, beta, alpha)
    qkv = torch.cat([q, k, v[..., v_storage_order().to(dev)]], dim=-1).contiguous().view(n * T, 3 * H)
    hh = h.clone().view(n * T, H)
    u = torch.full((n * T, H), float("nan"), dtype=torch.bfloat16, device=dev)
    rc = _lib.load().ditto_attn_self768(P(qkv), 3 * H, n, T, alpha, P(hh), P(gamma), P(beta), P(u) if with_ln else None, flags, ST())
    _lib.check(rc, "ditto_attn_self768")
    torch.cuda.synchronize()
    got_o = hh.view(n, T, H) - h
    return O.rel_l2(got_o.cpu(), want_o.cpu()), O.rel_l2(hh.view(n, T, H).cpu(), want_h.cpu()), \
        (O.rel_l2(u.float().view(n, T, H).cpu(), want_u.cpu()) if with_ln else 0.0), bool(torch.isfinite(hh).all())


@pytest.mark.parametrize("n,T", [(2, 750), (3, 1), (1, 100), (2, 128), (1, 129), (1, 257), (1, 375), (1, 2250), (1, 4096),
                                 (5, 40)])
def test_flash768_vs_torch(dev, n, T):
    eo, eh, eu, finite = run(dev, n, T)
    assert finite and eo <= 1e-2 and eh <= 3e-3 and eu <= 6e-3, (eo, eh, eu)


@pytest.mark.parametrize("n,T", [(70, 750), (200, 40), (150, 100), (12, 2250)])
def test_flash768_many_items_per_cluster(dev, n, T):
    """More work items than co-resident clusters: every cluster walks through several items, so the hand-overs between the
    epilogue of one item and the key loop of the next (TMEM, probability buffers, exchange slots, barrier phases) are exercised
    under load -- the single-item shapes above cannot see a hazard there.  Run twice: such hazards are timing dependent."""
    for seed in (0, 1):
        eo, eh, eu, finite = run(dev, n, T, seed=seed)
        assert finite and eo <= 1e-2 and eh <= 3e-3 and eu <= 6e-3, (seed, eo, eh, eu)


@pytest.mark.parametrize("n,T", [(2, 750), (1, 300), (1, 1500)])
def test_flash768_rescale_path(dev, n, T):
    """(i) forced: every tile that raises a row maximum rescales O in TMEM; (ii) provoked: keys scaled x4 per 128-key tile, so
    that later tiles exceed the reference by far more than the 2^8 laziness threshold; (iii) the two agree with the lazy run."""
    forced = run(dev, n, T, flags=1)
    assert forced[3] and forced[0] <= 1e-2 and forced[2] <= 6e-3, forced
    grow = lambda t: 4.0 ** (t // 128).float()   # noqa: E731
    lazy = run(dev, n, T, key_scale=grow, seed=3)
    both = run(dev, n, T, flags=1, key_scale=grow, seed=3)
    assert lazy[3] and lazy[0] <= 1e-2 and lazy[2] <= 6e-3, lazy
    assert both[3] and both[0] <= 1e-2 and both[2] <= 6e-3, both
    shrink = lambda t: 4.0 ** (-(t // 128).float())   # noqa: E731   (maxima fall: the reference never moves)
    down = run(dev, n, T, key_scale=shrink, seed=4)
    assert down[3] and down[0] <= 1e-2, down


def test_flash768_without_layernorm_stage(dev):
    eo, eh, _, finite = run(dev, 2, 200, with_ln=False)
    assert finite and eo <= 1e-2 and eh <= 3e-3


def test_flash768_rejects_bad_arguments(dev):
    lib = _lib.load()
    x = torch.zeros(8, 3 * H, dtype=torch.bfloat16, device=dev)
    hh = torch.zeros(8, H, device=dev)
    assert lib.ditto_attn_self768(None, 3 * H, 1, 8, 1.0, P(hh), None, None, None, 0, ST()) == -1
    assert lib.ditto_attn_self768(P(x), 3 * H, 1, 8, 1.0, P(hh), None, None, P(hh), 0, ST()) == -1     # LayerNorm output without gamma / beta
    assert lib.ditto_attn_self768(P(x), 100, 1, 8, 1.0, P(hh), None, None, None, 0, ST()) == -1          # row stride too small
