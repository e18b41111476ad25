"""Isolated launches of flash_attn768_kernel (ditto_attn_self768) for timing / ncu captures.
    python tools/attn768_bench.py [--n 32] [--T 750] [--iters 20] [--opt name=value]"""
import argparse
import ctypes as C
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from ditto_tts_b200 import _lib  # noqa: E402
from _opts import apply_opts  # noqa: E402

apply_opts()
ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=32)
ap.add_argument("--T", type=int, default=750)
ap.add_argument("--iters", type=int, default=20)
ap.add_argument("--flags", type=int, default=0, help="ditto_attn_self768 flags: bit 0 = always take the online-softmax rescale path")
ap.add_argument("--noln", type=int, default=0)
a = ap.parse_args()
dev = torch.device("cuda:0")
H = 768
P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
g = torch.Generator(device=dev).manual_seed(0)
qkv = torch.randn(a.n * a.T, 3 * H, device=dev, generator=g).bfloat16()
h = torch.randn(a.n * a.T, H, device=dev, generator=g)
u = torch.empty(a.n * a.T, H, dtype=torch.bfloat16, device=dev)
gamma, beta = torch.ones(H, device=dev), torch.zeros(H, device=dev)
lib = _lib.load()
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def run():
    _lib.check(lib.ditto_attn_self768(P(qkv), 3 * H, a.n, a.T, 1.0 / math.sqrt(H), P(h), P(gamma), P(beta), None if a.noln else P(u), a.flags, st))


for _ in range(3):
    run()
torch.cuda.synchronize()
ts = []
for _ in range(a.iters):
    flush.zero_()                       # L2 flush between timed launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run()
    e1.record()
    torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1) * 1e3)
ts.sort()
fl = 4.0 * a.T * a.T * H * a.n
print(f"flash768 n={a.n} T={a.T}: median {ts[len(ts) // 2]:.1f} us, best {ts[0]:.1f} us -> {fl / ts[len(ts) // 2] / 1e6:.0f} algorithmic TFLOP/s")
