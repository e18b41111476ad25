"""fp64 references of the DiT block sections, taken by their increment  --  TEST INFRASTRUCTURE ONLY.

The block sections (self-attention, cross-attention, gated MLP, DiT.py:103-139 / :141-148 / :150-155) each return
``x + f(x)``.  ``f(x)`` is only ~10 % of that sum's norm, so a bar on the sum lets defects of the attention pattern pass.
The tests therefore compare the increment ``out - x`` with the fp64 increment of the oracle.

This module holds what tests/test_gpu_section_increments.py (the CUDA kernels, -m gpu) and tests/test_section_sensitivity.py
(the CPU guard of the bars) share, so that the two cannot drift apart:

  * CASES, the bars and the seeded inputs of every case (optionally q / k projections sharpened so that softmax is peaked,
    optionally loud text tokens);
  * OFFSET_CASES: whole blocks whose rows carry a constant offset of ~1e3 times their spread.  LayerNorm is shift-invariant
    and every sublayer reads only LayerNorm outputs, so the offset leaves the reference increment unchanged; row statistics
    that cancel (fp32 E[v^2] - mean^2) do not;
  * the fp64 reference increments (the oracle's own functions, minus x);
  * a restatement of each section with the bf16 kernels' rounding points (bf16 operands u, W, q / k / v, the
    probabilities P, the attention output), which gives the error floor a correct kernel can reach;
  * planted defects of that restatement: what a kernel bug would do to the increment.  The guard asserts that each of
    them moves the checked error by a multiple of the bar.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

from . import ditto_oracle as O

Tensor = torch.Tensor

LAYER = 1                  # the block under test: layer 1 of a two-layer model, so a wrong layer index cannot pass
SHARP = 2.5                # q / k row scale of the sharpened cases: scores x 6.25, score std ~2 instead of ~0.33
WEIGHT_SEED, INPUT_SEED = 61, 62

# rel-L2 of the increment.  bf16: 7e-3 with the default weights (each row: 1.4e-2), 1.6e-2 for the attention sections with
# sharpened weights or loud text (the emulated floor is heavy-tailed per row there: no row bar).  The guard keeps floor <= bar / 2 and
# defect >= 2.5 bar.
BARS = {"bf16": 7e-3, "bf16_row": 1.4e-2, "bf16_sharp": 1.6e-2, "fp32": 1e-4}
FLOOR_MARGIN, DEFECT_MARGIN = 0.5, 2.5
SECTIONS = ("self", "cross", "mlp", "block")


@dataclass(frozen=True)
class Case:
    name: str
    hidden: int
    heads: int
    n: int
    T: int
    S: int
    sharp: bool = False          # q / k rows of both attentions x SHARP
    loud_text: bool = False      # text tokens 128.. with 4x the norm: the second key tile raises the row maxima
    sections: Tuple[str, ...] = SECTIONS
    fp32: bool = False           # also run the fp32 engine
    offset: float = 0.0          # |row offset| in [offset / 2, offset], sign mixed per row (0: none)
    const_text: bool = False     # every text row of a sequence equal (the constant-text path of the four-CTA kernel)


def _c(name, hidden, heads, n, T, S, **kw):
    return Case(name, hidden, heads, n, T, S, **kw)


CASES = (
    # one head of 768 (the product configuration): query / key tile edges of flash_attn768 (128 rows) and its four-CTA
    # variant (256 rows), the QKV + RoPE epilogue over many positions
    _c("t1", 768, 1, 3, 1, 40),
    _c("t127", 768, 1, 2, 127, 40),
    _c("t129", 768, 1, 2, 129, 40),
    _c("t256", 768, 1, 1, 256, 40),
    _c("t257", 768, 1, 2, 257, 40, fp32=True),
    _c("t750", 768, 1, 2, 750, 40),
    _c("t750_sharp", 768, 1, 2, 750, 40, sharp=True),
    _c("t2250", 768, 1, 1, 2250, 40),
    # max_seq_len: RoPE angles up to 4095 rad (inv_freq = 1), 32 key tiles, attention flatter than at any shorter length
    _c("t4096", 768, 1, 1, 4096, 40),
    # two of C5's own kernel combinations (parallel.c5_lengths): the two-CTA kernel with a partial 119-row query tile and
    # cross_fused; the four-CTA kernel over six query tiles and <CROSS> with exactly one full key tile
    _c("c5_t375_s32", 768, 1, 2, 375, 32),
    _c("c5_t1500_s128", 768, 1, 2, 1500, 128),
    # several work items per cluster / CTA: hand-over between consecutive items
    _c("load", 768, 1, 40, 750, 40, sections=("self", "cross")),
    # text lengths: cross_fused (S <= 64), flash_attn768q<CROSS> (64 < S <= 256), scores + softmax + P.V on the folded
    # path (256 < S <= 384), unfolded projections with the cluster scores + softmax kernel and row_lsum (S > 384)
    *(_c(f"s{S}", 768, 1, 2, 300, S, fp32=(S == 129)) for S in (1, 64, 65, 128, 129, 256, 257, 512)),
    *(_c(f"s{S}_sharp", 768, 1, 2, 300, S, sharp=True) for S in (1, 64, 65, 128, 129, 256, 257, 512)),
    # the second key tile of <CROSS> raises the row maxima far past the lazy-rescale threshold
    _c("s200_loud", 768, 1, 2, 300, 200, loud_text=True, sections=("cross",)),
    _c("s200_loud_sharp", 768, 1, 2, 300, 200, sharp=True, loud_text=True, sections=("cross",)),
    # twelve heads of 64: flash_attn_d64; S = 9 folded cross-attention, S = 100 unfolded
    *(_c(f"h12_t{T}_s{S}", 768, 12, 2, T, S, fp32=(T == 130 and S == 9)) for T in (130, 257, 750) for S in (9, 100)),
    _c("h12_t257_s100_sharp", 768, 12, 2, 257, 100, sharp=True),
    # generic epilogues (H not a multiple of 256 / several heads)
    _c("h256_t77", 256, 4, 2, 77, 9, fp32=True),
    _c("h256_t300", 256, 4, 2, 300, 33),
    _c("h256_t300_sharp", 256, 4, 2, 300, 33, sharp=True),
    _c("h128_t77", 128, 2, 2, 77, 5),
    _c("h128_t300", 128, 2, 2, 300, 20),
)
CASE = {c.name: c for c in CASES}
assert len(CASE) == len(CASES)

# whole blocks under a row offset, one per fused-LayerNorm site (tests/test_gpu_section_increments.py names the kernel each
# must reach).  bf16: |offset| <= 2048 keeps the fp32 rounding of h (ulp 2.4e-4) far below the bars.  fp32: the rounding of
# x + increment near the offset is itself ~1e-4 x offset / 1000 of the increment, so its offset is ~100.
OFFSET_CASES = (
    _c("off_t750", 768, 1, 2, 750, 40, sections=("block",), offset=2048.0),           # norm2: flash_attn768 / 768q
    _c("off_s64", 768, 1, 2, 300, 64, sections=("block",), offset=2048.0),            # norm3: cross_fused
    _c("off_s129", 768, 1, 2, 300, 129, sections=("block",), offset=2048.0),          # norm3: flash_attn768q<CROSS>
    _c("off_const", 768, 1, 2, 750, 40, sections=("block",), offset=2048.0, const_text=True),   # norm3: constant text
    _c("off_h12_s100", 768, 12, 2, 257, 100, sections=("block",), offset=2048.0),     # norm3: gemm_resid_ln after out_proj
    _c("off_s129_fp32", 768, 1, 2, 257, 129, sections=("block",), offset=128.0, fp32=True),
)
CASE.update({c.name: c for c in OFFSET_CASES})
assert len(CASE) == len(CASES) + len(OFFSET_CASES)
OFFSET_GUARD_CASES = ("off_t750", "off_h12_s100")

# the cases the CPU guard re-derives the bars on, each with its "_sharp" twin: every attention path of the table
GUARD_CASES = ("s64", "s129", "s257", "s512", "s200_loud", "h12_t257_s100", "h256_t300")
# cases whose floor the guard checks without planted defects: their paths are guard cases above, but not their lengths
# (the score-bias defect at S = 128, one key tile, moves the increment by only 2.05 bars: a guard case would need a twin)
FLOOR_CASES = ("t4096", "c5_t375_s32", "c5_t1500_s128")


def _peaked(case: Case, section: str) -> bool:
    """Attention with peaked softmax (sharpened q / k or loud text tokens): the heavy-tailed floor takes the larger bar.
    Neither changes the MLP."""
    return (case.sharp or case.loud_text) and section != "mlp"


def bar(case: Case, precision: str, section: str) -> float:
    if precision == "fp32":
        return BARS["fp32"]
    return BARS["bf16_sharp"] if _peaked(case, section) else BARS["bf16"]


def row_bar(case: Case, precision: str, section: str) -> Optional[float]:
    """Bar of the largest per-row error (None: not checked)."""
    return BARS["bf16_row"] if precision == "bf16" and not _peaked(case, section) else None


def twins(name: str):
    """A guard case and its sharpened twin: a defect counts as caught when one of the two clears the margin."""
    return tuple(CASE[k] for k in (name, name + "_sharp") if k in CASE)


def sharpen(sd: Dict[str, Tensor], layer: int, factor: float) -> Dict[str, Tensor]:
    """Scales the q and k rows of ``attn.in_proj_weight`` and ``cross_attn.in_proj_weight`` of block ``layer`` by
    ``factor`` (scores by factor^2), in a copy of the state dict."""
    sd = dict(sd)
    p = f"blocks.{layer}."
    H = sd[p + "norm1.weight"].numel()
    for key in ("attn.in_proj_weight", "cross_attn.in_proj_weight"):
        w = sd[p + key].clone()
        w[:2 * H] *= factor
        sd[p + key] = w
    return sd


def case_inputs(case: Case):
    """(cfg, fp32 state dict, x, text) of a case.  x is N(0, 1) around a N(0, 4^2) mean per row, so |mean| / spread stays
    below ~12: too small to expose cancelling row statistics, which is what OFFSET_CASES add (see row_offsets).  loud_text
    scales text tokens 128.. by 4; const_text repeats each sequence's first text row."""
    cfg = O.OracleConfig(case.hidden, 2, case.heads, 64, case.hidden, 50)
    sd = O.make_state_dict(cfg, WEIGHT_SEED)
    if case.sharp:
        sd = sharpen(sd, LAYER, SHARP)
    g = torch.Generator().manual_seed(INPUT_SEED)
    x = torch.randn(case.n, case.T, case.hidden, generator=g) + 4.0 * torch.randn(case.n, case.T, 1, generator=g)
    text = torch.randn(case.n, case.S, case.hidden, generator=g)
    if case.loud_text:
        text[:, 128:] *= 4.0
    if case.const_text:
        text = text[:, :1].expand_as(text).contiguous()
    if case.offset:
        x = (x.double() + row_offsets(case)).float()
    return cfg, sd, x, text


def row_offsets(case: Case) -> Tensor:
    """fp64 [n, T, 1] offsets added to x (fp32) by case_inputs: integers of either sign, |c| in [offset / 2, offset] (zeros
    without an offset).  ``x.double() - row_offsets(case)`` is exact, so the reference sees the input that was fed, unshifted."""
    if not case.offset:
        return torch.zeros(case.n, case.T, 1, dtype=torch.float64)
    g = torch.Generator().manual_seed(INPUT_SEED + 1)
    mag = torch.round(case.offset * (1 + torch.rand(case.n, case.T, 1, generator=g, dtype=torch.float64)) / 2)
    sign = torch.where(torch.rand(case.n, case.T, 1, generator=g) < 0.5, -1.0, 1.0).double()
    return sign * mag


def _f64(sd, x, text):
    return {k: v.double() for k, v in sd.items()}, x.double(), text.double()


def increments(case: Case, sd, x, text) -> Dict[str, Tensor]:
    """fp64 increments ``section(x) - x`` of the oracle for the case's sections ("block": the whole DiT block).  The row
    offsets of the case are taken off x first: the sections are shift-invariant, so this is the increment of x itself,
    computed without the offset's cancellation."""
    sd, x, text = _f64(sd, x, text)
    x = x - row_offsets(case)
    rot = O.rotary_angles(case.T, case.hidden // case.heads, torch.float64)
    p = f"blocks.{LAYER}."
    f = {"self": lambda: O.self_attention(sd, p, x, rot, case.heads),
         "cross": lambda: O.cross_attention(sd, p, x, text, case.heads),
         "mlp": lambda: O.gated_mlp(sd, p, x),
         "block": lambda: O.dit_block(sd, LAYER, x, text, rot, case.heads)}
    return {s: f[s]() - x for s in case.sections}


def errors(got: Tensor, want: Tensor) -> Tuple[float, float]:
    """(rel-L2 over the whole tensor, largest rel-L2 of one row) of an increment against the reference increment."""
    got, want = got.double().cpu(), want.double().cpu()
    rows = (got - want).flatten(0, -2).norm(dim=-1) / want.flatten(0, -2).norm(dim=-1).clamp_min(1e-300)
    return O.rel_l2(got, want), float(rows.max())


# ------------------------------------------------------------------------------------------------------------------------
# restatement with the kernels' bf16 rounding points, and planted defects
# ------------------------------------------------------------------------------------------------------------------------
DEFECTS = {
    "self": ("rope_shifted_one_row", "rope_missing", "rope_interleaved_pairs", "keys_from_256_ignored", "mean_of_v",
             "v_columns_swapped"),
    "cross": ("mean_of_v", "score_bias_dropped", "last_token_ignored"),
    "mlp": ("hidden_columns_swapped", "gelu_tanh"),
}
# kept to record what bf16 cannot see: its effect (~2e-4) is below the rounding of an increment, it is not a checked defect
INVISIBLE = {("mlp", "gelu_tanh")}
# norm2 and norm3 with one-pass fp32 statistics (_ln_one_pass_fp32), planted in a whole block: only a row offset makes it
# visible (at the |mean| / spread <= ~12 of CASES it moves an increment by ~1e-5), so only OFFSET_CASES are checked for it
OFFSET_DEFECT = ("block", "layernorm_one_pass_fp32")


def _bf(z: Tensor) -> Tensor:
    return z.to(torch.bfloat16).to(z.dtype)


def _ln_one_pass_fp32(x, w, b):
    """LayerNorm with fp32 one-pass statistics var = E[v^2] - mean^2 in the partial-sum order of gemm_resid_ln's epilogue:
    column parts of 128, each 4 threads x 32 serial (fused) multiply-adds, then the 4-thread sums and the parts in turn.
    Wrong by ~eps (mean / spread)^2 in the variance: the defect a cancelling row-statistics kernel makes."""
    H = x.shape[-1]
    assert H % 128 == 0
    v = x.float().reshape(*x.shape[:-1], H // 128, 4, 32)
    s = torch.zeros(v.shape[:-1], dtype=torch.float32)
    q = torch.zeros_like(s)
    for k in range(32):                       # fp32 sum; fma: exact product (fp64) + one rounding to fp32
        s = s + v[..., k]
        q = (v[..., k].double() ** 2 + q.double()).float()
    s, q = s.sum(-1), q.sum(-1)               # 4-thread (quad) sums in fp32
    S, Q = s[..., 0], q[..., 0]
    for c in range(1, H // 128):
        S, Q = S + s[..., c], Q + q[..., c]
    inv_n = torch.tensor(1.0 / H, dtype=torch.float32)
    mean = S * inv_n
    rstd = torch.rsqrt(torch.clamp_min(Q * inv_n - mean * mean, 0.0) + 1e-5)
    return (x - mean.double()[..., None]) * rstd.double()[..., None] * w + b


def _ln(x, w, b, one_pass):
    return _ln_one_pass_fp32(x, w, b) if one_pass else F.layer_norm(x, (x.shape[-1],), w, b, 1e-5)


def _self(sd, p, x, heads, rot, r, defect):
    n, T, H = x.shape
    d = H // heads
    u = r(F.layer_norm(x, (H,), sd[p + "norm1.weight"], sd[p + "norm1.bias"], 1e-5))
    w, b = r(sd[p + "attn.in_proj_weight"]), sd[p + "attn.in_proj_bias"]
    q, k, v = (F.linear(u, w[i * H:(i + 1) * H], b[i * H:(i + 1) * H]).reshape(n, T, heads, d) for i in range(3))
    if defect == "rope_shifted_one_row":
        rot = torch.roll(rot, 1, 0)
    if defect == "rope_missing":
        rot = torch.zeros_like(rot)
    if defect == "rope_interleaved_pairs":      # (2i, 2i+1) pairs instead of rotate_half's (i, i + d/2)
        c = torch.repeat_interleave(rot[:, :d // 2], 2, -1)[None, :, None]
        pair = lambda z: torch.stack([-z[..., 1::2], z[..., 0::2]], -1).flatten(-2)  # noqa: E731
        q, k = q * c.cos() + pair(q) * c.sin(), k * c.cos() + pair(k) * c.sin()
    else:
        q, k = O.apply_rope(rot, q), O.apply_rope(rot, k)
    q, k, v = (r(z).permute(0, 2, 1, 3) for z in (q, k, v))
    s = q @ k.transpose(-1, -2) / math.sqrt(d)
    if defect == "keys_from_256_ignored":
        s[..., 256:] = -math.inf
    P = torch.exp(s - s.amax(-1, keepdim=True))              # unnormalised P in bf16, the row sum in fp32
    o = (r(P) @ v) / P.sum(-1, keepdim=True)
    if defect == "mean_of_v":
        o = v.mean(-2, keepdim=True).expand_as(o)
    o = o.permute(0, 2, 1, 3).reshape(n, T, H)
    if defect == "v_columns_swapped":
        o = o[..., [1, 0] + list(range(2, H))]
    return o


def _cross(sd, p, x, text, heads, r, defect, ln_one_pass=False):
    n, T, H = x.shape
    S, d = text.shape[1], H // heads
    u = r(_ln(x, sd[p + "norm2.weight"], sd[p + "norm2.bias"], ln_one_pass))
    w, b = sd[p + "cross_attn.in_proj_weight"], sd[p + "cross_attn.in_proj_bias"]
    bq = torch.zeros_like(b[:H]) if defect == "score_bias_dropped" else b[:H]   # folded: the score bias sqrt(1/d) bq.k_j
    q = F.linear(u, r(w[:H]), bq).reshape(n, T, heads, d).permute(0, 2, 1, 3)
    k = r(F.linear(text, w[H:2 * H], b[H:2 * H])).reshape(n, S, heads, d).permute(0, 2, 1, 3)
    v = r(F.linear(text, w[2 * H:], b[2 * H:])).reshape(n, S, heads, d).permute(0, 2, 1, 3)
    s = (q @ k.transpose(-1, -2)) / math.sqrt(d)
    if defect == "last_token_ignored":
        s[..., -1] = -math.inf
    o = r(torch.softmax(s, -1)) @ v
    if defect == "mean_of_v":
        o = v.mean(-2, keepdim=True).expand_as(o)
    o = o.permute(0, 2, 1, 3).reshape(n, T, H)
    return F.linear(r(o), r(sd[p + "cross_attn.out_proj.weight"]), sd[p + "cross_attn.out_proj.bias"])


def _mlp(sd, p, x, r, defect, ln_one_pass=False):
    H = x.shape[-1]
    u = r(_ln(x, sd[p + "norm3.weight"], sd[p + "norm3.bias"], ln_one_pass))
    a = F.linear(u, r(sd[p + "mlp_fc1.weight"]), sd[p + "mlp_fc1.bias"])
    gate = F.linear(u, r(sd[p + "gate.weight"]), sd[p + "gate.bias"])
    g = F.gelu(a, approximate="tanh" if defect == "gelu_tanh" else "none") * torch.sigmoid(gate)
    if defect == "hidden_columns_swapped":
        g = g[..., [1, 0] + list(range(2, 4 * H))]
    return F.linear(r(g), r(sd[p + "mlp_fc2.weight"]), sd[p + "mlp_fc2.bias"])


def restated(case: Case, sd, x, text, section: str, bf16: bool = False, defect: Optional[Tuple[str, str]] = None) -> Tensor:
    """fp64 increment of ``section`` from the restatement above: with the kernels' bf16 rounding points (bf16=True) and / or
    one planted defect (section, name).  "block" chains the three sections, the defect landing in its own section (a "block"
    defect in norm2 and norm3), and with bf16=True keeps the residual stream in fp32 as the kernels do.  x is what was fed,
    row offsets included."""
    sd, x, text = _f64(sd, x, text)
    rot = O.rotary_angles(case.T, case.hidden // case.heads, torch.float64)
    p = f"blocks.{LAYER}."
    r = _bf if bf16 else (lambda z: z)
    dd = lambda s: defect[1] if defect is not None and defect[0] == s else None  # noqa: E731
    one_pass = defect == OFFSET_DEFECT
    f = {"self": lambda h: _self(sd, p, h, case.heads, rot, r, dd("self")),
         "cross": lambda h: _cross(sd, p, h, text, case.heads, r, dd("cross"), one_pass),
         "mlp": lambda h: _mlp(sd, p, h, r, dd("mlp"), one_pass)}
    if section != "block":
        return f[section](x)
    h = x
    for s in ("self", "cross", "mlp"):
        h = h + f[s](h)
        if bf16:
            h = h.float().double()
    return h - x
