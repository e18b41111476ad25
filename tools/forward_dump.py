"""Plain-context forwards on every cross-attention path (the cases of tests/test_gpu_text_mask.py), saved to one file, so
that two builds of the library can be compared bit for bit:

    python tools/forward_dump.py --out new.pt
    python tools/forward_dump.py --lib /path/to/other/libditto_b200.so --out old.pt
    python tools/forward_dump.py --compare old.pt new.pt      # prints one JSON line: bitwise equality per case
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _opts import apply_opts  # noqa: E402

apply_opts()   # --lib path: a differently built library
ap = argparse.ArgumentParser()
ap.add_argument("--out")
ap.add_argument("--compare", nargs=2)
a = ap.parse_args()

if a.compare:
    x, y = (torch.load(p) for p in a.compare)
    same = {k: bool(torch.equal(x[k], y[k])) for k in sorted(x)}
    print(json.dumps({"bitwise_equal": same, "all": all(same.values()) and set(x) == set(y)}))
    sys.exit(0)

import ditto_tts_b200 as D  # noqa: E402
from ditto_tts_b200 import _lib  # noqa: E402
import ctypes  # noqa: E402

# an older build may predate symbols this package declares; the plain forward needs none of those
_other = ctypes.CDLL(_lib.LIB_PATH)
for _name in [n for n in _lib.SIGNATURES if not hasattr(_other, n)]:
    del _lib.SIGNATURES[_name]
from oracle import ditto_oracle as O  # noqa: E402

# name -> (hidden, heads, precision, engine switches, DiTTO keywords, T, S)
CASES = {
    "cross_fused": (768, 1, "bf16", {}, {}, 750, 64),
    "cross_flash": (768, 1, "bf16", {}, {}, 750, 192),
    "folded_scores_300": (768, 1, "bf16", {}, {}, 150, 300),
    "unfolded_two_tile_512": (768, 1, "bf16", {}, {}, 150, 512),
    "multihead_folded": (256, 4, "bf16", {}, {}, 150, 24),
    "multihead_unfolded": (256, 4, "bf16", {}, {}, 150, 48),
    "fp32": (768, 1, "fp32", {}, {}, 150, 64),
    "no_fused_cross": (768, 1, "bf16", {"no_fused_cross": 1}, {}, 150, 64),
    "no_cross_flash": (768, 1, "bf16", {"no_cross_flash": 1}, {}, 150, 192),
    "unfused_softmax_400": (768, 1, "bf16", {}, {"fused_attn": False}, 150, 400),
}
dev = torch.device("cuda:0")
out = {}
for name, (H, heads, prec, opts, kw, T, S) in CASES.items():
    cfg = O.OracleConfig(H, 2, heads, 256, H, 20)
    m = D.DiTTO(hidden_dim=H, num_layers=2, num_heads=heads, time_dim=256, text_dim=H, diffusion_steps=20, precision=prec, **kw)
    m.load_state_dict(O.make_state_dict(cfg, 91 + H + heads), strict=True)
    m = m.to(dev)
    for k, v in opts.items():
        _lib.debug_option(k, v)
    try:
        m.engine()
    finally:
        _lib.debug_option("reset", 0)
    g = torch.Generator().manual_seed(5)
    B = 3
    x, text = torch.randn(B, T, H, generator=g), torch.randn(B, S, H, generator=g)
    text[2] = text[2, :1]          # a constant text
    t = torch.randint(0, 20, (B,), generator=g)
    both = torch.cat([text, torch.zeros_like(text)]).to(dev)   # with the zero null text of CFG
    ctx = m.text_context(both, T_hint=T)
    out[name] = m.forward_with_context(x.to(dev), ctx, torch.cat([t, t]).to(dev), 2 * B, S).cpu()
    del m
torch.save(out, a.out)
print(json.dumps({"saved": a.out, "cases": len(out)}))
