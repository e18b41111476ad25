"""Cost of a sampling job by sampler: DDPM over all 50 timesteps (the bench path) against DDIM and DPM-Solver++(2M) over
K in {10, 16, 25} visited timesteps, eta in {0, 1}, on one GPU.

    python tools/sampler_steps.py [--batches 256,16,1] [--ks 10,16,25] [--repeats 2] [--prompt-frames P]

Model and inputs are bench.py's (repo-default DiT, H = 768, L = 5, one head, bf16, random init from torch.manual_seed(0);
10 s utterances, T = 750 frames, S = 64 text tokens, CFG w = 3, noise drawn in the update kernel), with a 50-step
schedule.  A job is what DiTTOSampler.sample_latents runs on its graph path: reset, then per visited timestep the t fill
(sub-sequences only) and one CUDA-graph replay; it is timed with CUDA events, inputs resident in HBM.  Every configuration
is timed once per round, in the same order every round, on the same GPU (--repeats rounds); ms_per_job is the median.
The update kernel's class time and bytes come from the library profiler over 3 eager steps (ditto_profile_*).  The card's
name, power limit and the SM clock sampled during each timed job are printed beside the numbers.

With --prompt-frames P every sampler also runs a prompted job: the first P frames of every utterance are known latents
(sample_latents(..., known=, known_mask=), a speech prompt of P / 75 s), timed alternately with the unprompted one.

One JSON line per (batch, sampler); batch 256 is C4, 16 is C2, 1 is the single-utterance latency (bench's
rtf.single_utterance shape)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import bench  # noqa: E402
import ditto_tts_b200 as D  # noqa: E402
from ditto_tts_b200 import _lib  # noqa: E402
from ditto_tts_b200.model import _ptr, _stream  # noqa: E402

DIFFUSION_STEPS = 50


def card():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        name, plim, smax = (c.strip() for c in r.stdout.strip().split(","))
        return {"name": name, "power_limit_w": float(plim), "sm_max_mhz": float(smax)}
    except Exception:  # noqa: BLE001  (nvidia-smi missing: the numbers are still the GPU's, only unlabelled)
        return {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}


class Job:
    def __init__(self, model, method, K, eta, B, dev, seed, prompt=0):
        kw = {} if method == "ddpm" else dict(method=method, num_steps=K, eta=eta)
        self.name = f"{method}-{K}" + ("" if method == "ddpm" else f" eta={eta:g}") + (f" prompt={prompt}" if prompt else "")
        self.method, self.K, self.eta, self.B, self.prompt = method, K, eta, B, prompt
        self.s = D.DiTTOSampler(model, guidance_scale=bench.GUIDANCE, **kw)
        self.s._activate(known=prompt > 0)
        g = torch.Generator().manual_seed(seed)
        self.text = torch.randn(B, bench.TEXT_LEN, bench.HIDDEN, generator=g).to(dev)
        self.x0 = torch.randn(B, bench.FRAMES_10S, bench.HIDDEN, generator=g).to(dev)
        self.known = self.mask = None
        if prompt:                           # the prompt's latents: known frames 0 .. P-1 of every utterance
            self.known = torch.randn(B, bench.FRAMES_10S, bench.HIDDEN, generator=g).to(dev)
            self.mask = torch.zeros(B, bench.FRAMES_10S, dtype=torch.uint8, device=dev)
            self.mask[:, :prompt] = 1
            self.x0 = self.s._known_start(self.x0, self.known, self.mask)
        self.ctx = self.s._context(self.text, True, None, bench.FRAMES_10S)
        self.g = self.s.step_graph(B, bench.FRAMES_10S, bench.TEXT_LEN, True, bench.GUIDANCE, self.ctx, True, dev, known=prompt > 0)
        self.taus = self.s.timesteps.tolist()
        self.consecutive = K == DIFFUSION_STEPS
        self.seed = seed

    def activate(self):
        self.s._activate(known=self.prompt > 0)

    def run(self):
        """One job, the loop of DiTTOSampler.sample_latents' graph path."""
        self.g.reset(self.x0, self.taus[0], self.seed, known=self.known, known_mask=self.mask)
        for t in self.taus:
            if not self.consecutive:
                self.g.t.fill_(t)
            self.g.replay()

    def eager_profile(self, steps=3):
        g, lib = self.g, _lib.load()
        g.reset(self.x0, self.taus[0], self.seed, known=self.known, known_mask=self.mask)
        torch.cuda.synchronize()
        _lib.profile_start()
        for t in self.taus[:steps]:
            g.t.fill_(t)
            args = (self.s.model.engine(), _ptr(g.x), _ptr(g.ctx), _ptr(g.t), _ptr(g.rng), 1, bench.GUIDANCE, self.B,
                    bench.FRAMES_10S, bench.TEXT_LEN, _ptr(g.eps), _ptr(g.x))
            if g.known is not None:
                _lib.check(lib.ditto_p_sample_known(*args[:4], None, *args[4:], _ptr(g.hist), _ptr(g.known), _ptr(g.mask), _ptr(g.ws),
                                                    g.ws.numel(), 1, _stream()))
            elif g.hist is not None:
                _lib.check(lib.ditto_p_sample_multistep_rng(*args, _ptr(g.hist), _ptr(g.ws), g.ws.numel(), 1, _stream()))
            else:
                _lib.check(lib.ditto_p_sample_rng(*args, _ptr(g.ws), g.ws.numel(), 1, _stream()))
        prof = _lib.profile_stop()
        torch.cuda.synchronize()
        upd = prof.get("cfg_ddpm_update", {"ms": 0.0, "bytes": 0.0, "launches": 0})
        return {"update_ms_per_step": upd["ms"] / steps, "update_bytes_per_step": upd["bytes"] / steps,
                "update_bytes_per_element": upd["bytes"] / steps / (self.B * bench.FRAMES_10S * bench.HIDDEN),
                "update_launches_per_step": upd["launches"] // steps,
                "profiled_step_ms": sum(v["ms"] for v in prof.values()) / steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,16,1")
    ap.add_argument("--ks", default="10,16,25")
    ap.add_argument("--etas", default="0,1")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--prompt-frames", type=int, default=0, help="also time every sampler with this many known leading frames")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sampler_steps.py: no CUDA device (the product path has no CPU fallback)")
    dev = torch.device("cuda:0")
    info = card()
    clocks = bench.ClockSampler(0).start()
    torch.manual_seed(0)
    model = D.DiTTO(hidden_dim=bench.HIDDEN, num_layers=bench.LAYERS, num_heads=bench.HEADS, time_dim=bench.TIME_DIM,
                    text_dim=bench.HIDDEN, diffusion_steps=DIFFUSION_STEPS, precision="bf16").to(dev)
    ks = [int(k) for k in a.ks.split(",")]
    etas = [float(e) for e in a.etas.split(",")]
    specs = [("ddpm", DIFFUSION_STEPS, 0.0)] + [(m, k, e) for m in ("ddim", "dpmpp_2m") for k in ks for e in etas]
    for B in (int(b) for b in a.batches.split(",")):
        prompts = [0] + ([a.prompt_frames] if a.prompt_frames > 0 else [])
        jobs = [Job(model, m, k, e, B, dev, 1, p) for m, k, e in specs for p in prompts]   # unprompted / prompted alternate
        times = {j.name: [] for j in jobs}
        clk = {j.name: [] for j in jobs}
        for j in jobs:                       # warm-up: one job each (graphs were captured when built)
            j.activate()
            j.run()
        torch.cuda.synchronize()
        for _ in range(a.repeats):
            for j in jobs:
                j.activate()                 # samplers share the model: the engine takes this one's tables (host, untimed)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                w0 = time.perf_counter()
                e0.record()
                j.run()
                e1.record()
                torch.cuda.synchronize()
                w1 = time.perf_counter()
                times[j.name].append(e0.elapsed_time(e1))
                clk[j.name].append(clocks.summary(w0, w1).get("sm_mhz"))
        base = statistics.median(times[jobs[0].name])
        for j in jobs:
            j.activate()
            prof = j.eager_profile()
            ms_job = statistics.median(times[j.name])
            finite = bool(torch.isfinite(j.g.x).all())
            line = {"tool": "sampler_steps", "batch": B, "T": bench.FRAMES_10S, "S": bench.TEXT_LEN,
                    "shape": {256: "C4", 16: "C2", 1: "single 10 s utterance"}.get(B, f"B={B}"),
                    "sampler": j.method, "steps": j.K, "eta": j.eta, "prompt_frames": j.prompt,
                    "ms_per_job": ms_job, "ms_per_step": ms_job / j.K,
                    "ms_per_job_runs": times[j.name], "job_vs_ddpm50": ms_job / base,
                    "launches_per_step": int(j.g.launches_per_step), **prof,
                    "sm_mhz_per_run": clk[j.name], "gpu": info, "outputs_finite": finite}
            print(json.dumps(line), flush=True)
        del jobs
        torch.cuda.empty_cache()
    clocks.stop()


if __name__ == "__main__":
    main()
