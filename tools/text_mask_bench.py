"""Per-utterance text lengths on a realistic text mix: C5's 256 durations (parallel.c5_lengths) with every token count
jittered by u ~ U(0.8, 1.25), so S no longer follows T.  50-step DDPM, CFG w = 3, seeded, bf16, H = 768, 5 layers.

  A  exact texts: one ragged group per distinct (T, S) pair
  B  texts zero-padded to 64 / 128 / 256 tokens with text_lengths: one group per (T, padded width)

Per arm: ms per step (CUDA events around the replays of one captured step graph; arms alternated), launches per step, group
count, and over three successive jobs with fresh jitter and the same T multiset the graph captures and the host time of
each job.  Also the largest per-utterance rel-L2 between the arms.  A second measurement times a uniform B = 16, T = 750
batch with a plain S = 64 context against S_pad = 64 with lengths drawn in [8, 64].

    python tools/text_mask_bench.py [--repeats 3] [--steps 50] [--opt name=value] [--lib path]
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ditto_tts_b200 as D  # noqa: E402
from ditto_tts_b200 import parallel, ragged  # noqa: E402
from ditto_tts_b200.ragged import RaggedBatch, RaggedStepGraph  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from _opts import apply_opts  # noqa: E402

apply_opts()
ap = argparse.ArgumentParser()
ap.add_argument("--utts", type=int, default=256)
ap.add_argument("--steps", type=int, default=50)
ap.add_argument("--repeats", type=int, default=3)
ap.add_argument("--layers", type=int, default=5)
a = ap.parse_args()

dev = torch.device("cuda:0")
H, K, W = 768, a.steps, 3.0
BUCKETS = (64, 128, 256)


def card():
    name = torch.cuda.get_device_name(dev)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def jittered(seed):
    """C5 frames with the token counts jittered by u ~ U(0.8, 1.25) under random.Random(seed)."""
    T, S = parallel.c5_lengths(a.utts)
    rnd = random.Random(seed)
    return T, [max(1, int(round(s * rnd.uniform(0.8, 1.25)))) for s in S]


def bucket(s):
    return next(b for b in BUCKETS if s <= b)


def arm_inputs(T, S, exact, g):
    texts = [torch.randn(s, H, generator=g) for s in S]
    if exact:
        return [x.to(dev) for x in texts], None
    padded = []
    for x in texts:
        p = torch.zeros(bucket(x.shape[0]), H)
        p[:x.shape[0]] = x
        padded.append(p.to(dev))
    return padded, list(S)


torch.manual_seed(0)
m = D.DiTTO(hidden_dim=H, num_layers=a.layers, num_heads=1, time_dim=256, text_dim=H, diffusion_steps=K, precision="bf16").to(dev)
T1, S1 = jittered(1)
seeds = list(range(1000, 1000 + a.utts))
res = {"workload": f"jittered C5: {a.utts} utterances, {sum(T1)} frames, {K}-step DDPM, CFG w = {W}, bf16, H = {H}, L = {a.layers}"}
res["card"], res["power_limit"] = card()

# ---- ms per step, arms alternated on one captured step graph each
graphs, outs = {}, {}
for name, exact in (("A_exact", True), ("B_padded", False)):
    texts, lens = arm_inputs(T1, S1, exact, torch.Generator().manual_seed(7))
    rb = RaggedBatch(m, texts, T1, guided=True, text_lengths=lens)
    s = D.DiTTOSampler(m, W)
    outs[name] = s.sample_latents_ragged(texts, T1, seeds=seeds, text_lengths=lens)   # also the cross-arm difference
    graphs[name] = (rb, RaggedStepGraph(rb, W, True))
x0 = {k: torch.randn(rb.x_rows, H, device=dev) for k, (rb, _) in graphs.items()}


def timed(g, x):
    g.reset(x, K - 1, seed=1)
    for _ in range(3):
        g.replay()
    g.reset(x, K - 1, seed=1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K


times = {k: [] for k in graphs}
for _ in range(a.repeats):
    for k, (rb, g) in graphs.items():
        times[k].append(timed(g, x0[k]))
for k, (rb, g) in graphs.items():
    res[k] = {"ms_per_step": sorted(times[k]), "launches_per_step": g.launches_per_step, "groups": len(rb.groups)}
res["max_rel_l2_between_arms"] = max(float((p - q).norm() / q.norm()) for p, q in zip(outs["A_exact"], outs["B_padded"]))
del graphs

# ---- three successive jobs with fresh jitter and the same T multiset: captures and host time
captures = [0]
_init = RaggedStepGraph.__init__


def counting_init(self, *args, **kw):
    captures[0] += 1
    _init(self, *args, **kw)


ragged.RaggedStepGraph.__init__ = counting_init
for name, exact in (("A_exact", True), ("B_padded", False)):
    s = D.DiTTOSampler(m, W)
    captures[0] = 0
    host = []
    for j in range(3):
        T, S = jittered(2 + j)
        texts, lens = arm_inputs(T, S, exact, torch.Generator().manual_seed(20 + j))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s.sample_latents_ragged(texts, T, seeds=seeds, text_lengths=lens)
        torch.cuda.synchronize()
        host.append(round(time.perf_counter() - t0, 3))
    res[name].update({"captures_over_3_jobs": captures[0], "job_seconds": host})
ragged.RaggedStepGraph.__init__ = _init

# ---- uniform B = 16, T = 750: plain S = 64 against S_pad = 64 with lengths in [8, 64]
B, T, S = 16, 750, 64
g = torch.Generator().manual_seed(9)
text = torch.randn(B, S, H, generator=g).to(dev)
lens = torch.randint(8, S + 1, (B,), generator=g).tolist()
xu = torch.randn(B, T, H, generator=g).to(dev)
uni = {}
both = torch.cat([text, torch.zeros_like(text)])          # [cond; uncond], the sampler's layout
for name, ln in (("plain_S64", None), ("masked_S64", lens)):
    s = D.DiTTOSampler(m, W)
    ctx = m.text_context(both, name=f"bench_{name}", T_hint=T, text_lengths=None if ln is None else ln + ln)   # one buffer each
    uni[name] = (s.step_graph(B, T, S, True, W, ctx, True, dev), s)
ut = {k: [] for k in uni}
for _ in range(a.repeats):
    for k, (sg, _) in uni.items():
        ut[k].append(timed(sg, xu))
res["uniform_B16_T750"] = {k: {"ms_per_step": sorted(v), "launches_per_step": uni[k][0].launches_per_step} for k, v in ut.items()}
res["uniform_B16_T750"]["lengths"] = lens
print(json.dumps(res))
