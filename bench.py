#!/usr/bin/env python
"""bench.py -- headline benchmark of the DiTTo-TTS denoiser hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Model: the repo-default DiT (hidden 768, 5 layers, 1 head of 768, time 256; src/utils/Config.py:109-113), random-init
weights, bf16 tensor-core path with fp32 accumulation / residual stream / statistics.  A "step" is one denoising step of
DDPM sampling with classifier-free guidance (w = 3, unconditional = zero text embedding): one forward over 2B sequences
(conditional + unconditional sharing x) + the fused CFG-combine / DDPM-update kernel that also draws the step's noise.
K steps = one full sampling job with DIFFUSION_STEPS = K (the reference's own way of choosing the step count).

Workloads (BASELINE.json configs):
  c4 (default) 256 x 10 s utterances (T = 750 frames, S = 64 text tokens) sharded by utterance over the N GPUs -- 256 / N per
               GPU, STRONG scaling, no collective inside a step, one NCCL all_gather of the final latents afterwards.  This
               is the configuration the metric ("latent frames/sec per denoising step at 1/2/4/8 B200") is quoted on; it
               fits one GPU (11 GB of workspace), so N = 1 runs all 256.
  c2           16 x 10 s utterances per GPU (weak scaling); at N = 1 its numbers are also reported under "c2" in the c4 line
  c3           4 x 30 s utterances per GPU (T = 2250, S = 192; attention-dominated)
  c5           256 utterances of 2-20 s (random.seed(0) durations, T = 75 s, S = round(6.4 s)), every one at its own length
               (packed, unpadded), balanced by cost over the N GPUs; value counts VALID frames

value   = latent frames / s per denoising step = (frames of all utterances on all GPUs) / (time of one step), inputs
          resident in HBM.  The timed region is one K-step job: exactly K = --steps steps after the W warm-up steps.
--dump-outputs DIR writes, after the timed region, the final latents of that job on rank 0 (what sample_latents returns)
          as DIR/latents.npy, float32 [frames, 768]: all frames, or a fixed seeded sample of DUMP_ROWS frames in frame order
          when there are more.  Weights, inputs and the job's noise seed are fixed, so two builds compare row for row.
e2e     = the same metric through the public API (DiTTOSampler.sample_latents) starting from PINNED HOST text embeddings
          and x_T and ending with the final latents back in host memory; copies are inside the timed region.
roofline= the dominant kernel class timed live with CUDA events on the launching stream (library profiler, eager steps
          after the timed region): algorithmic flops / measured peak.  Denominator: the burst bf16 figure of
          MEASURED_PEAKS.json when the SM clock sampled during the timed region stayed near its maximum, the sustained one
          when it sagged; both fractions are printed.  `traffic` is an ncu figure and is only reported when
          profiles/traffic.json was captured from exactly this kernel source (sha of csrc/), else null.
cpu_baseline / --impl reference = the reference's own CPU implementation (oracle/_ref = its DiT.py / DiTTO.py, imported
          unmodified; falls back to the oracle port) on all host threads, on a bounded sample: CFG steps of ONE utterance.
Parity bars (tests/, BASELINE.json): rel-L2 <= 2e-2 (bf16 path) and <= 1e-4 (fp32 path) vs the fp32 reference.
"""
from __future__ import annotations

import argparse
import atexit
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HIDDEN, LAYERS, HEADS, TIME_DIM = 768, 5, 1, 256
FRAMES_10S, TEXT_LEN, GUIDANCE = 750, 64, 3.0
C4_UTTERANCES = 256
DUMP_ROWS = 16384   # 48 MiB of float32 frames at H = 768: a --dump-outputs directory stays under 64 MB


def forward_flops(T, S):
    """SURVEY.md 8a: algorithmic flops per sequence per forward (dead self-attn out_proj excluded)."""
    H, L = HIDDEN, LAYERS
    return L * (34.0 * T * H * H + 4.0 * T * T * H + 4.0 * T * S * H) + 4.0 * T * H * H


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(burst=float(d["bf16_tflops"]), sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    hbm=float(d["hbm_gbs"]), source="measured (MEASURED_PEAKS.json)")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def choose_peak(peaks, clocks):
    """Burst figure when the sampled SM clock stayed within 7 % of its maximum during the timed region (a short region,
    or a box that holds its clock), the sustained figure when it sagged (a long region at the power cap)."""
    sm, mx = clocks.get("sm_mhz"), clocks.get("sm_max_mhz")
    if sm and mx and sm < 0.93 * mx:
        return "sustained", peaks["sustained"]
    return "burst", peaks["burst"]


def csrc_sha():
    """sha256 over the CUDA sources: ties an ncu-derived number in profiles/ to the code it was captured from."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "ditto_tts_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh")):
            with open(os.path.join(d, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def traffic_for(kernel_class):
    """DRAM bytes per launch from the committed `ncu --set full` capture -- only if it was taken from this source tree."""
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(tp):
        return None, "no capture"
    with open(tp) as f:
        t = json.load(f)
    if t.get("_csrc_sha") != csrc_sha():
        return None, "capture predates the current kernel source (profiles/traffic.json _csrc_sha differs)"
    v = t.get(kernel_class)
    return (float(v) if v is not None else None), t.get("_source", "profiles/traffic.json")


def per_class_roofline(prof, peak_tflops, peak_gbs):
    """Every kernel class of the profiled steps against ITS roofline: the bound is whichever of (algorithmic flops / tensor peak)
    and (algorithmic bytes / HBM copy peak) takes longer, `frac` = that time / the measured time.  Flops and bytes are what the
    launchers declare (SURVEY 8d: no credit for padding rows; bytes = the tensors a launch must read and write once)."""
    out = {}
    for name, v in sorted(prof.items()):
        t = v["ms"] / 1e3
        if t <= 0.0:
            continue
        t_tensor = v["flops"] / (peak_tflops * 1e12) if v["flops"] else 0.0
        t_hbm = v["bytes"] / (peak_gbs * 1e9) if v["bytes"] else 0.0
        bound = "tensor" if t_tensor >= t_hbm else "hbm"
        ach = v["flops"] / t / 1e12 if bound == "tensor" else v["bytes"] / t / 1e9
        out[name] = {"bound": bound, "achieved": round(ach, 1), "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                     "frac": round(max(t_tensor, t_hbm) / t, 3)}
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms.  Started well before the timed region (nvidia-smi needs up
    to a second to come up on an 8-GPU box); summary() keeps the samples whose arrival time falls inside the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            atexit.register(self.stop)   # never leave the sampler behind, whatever path the bench exits through
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, t0, t1):
        """Samples that arrived in [t0, t1 + one period]; when the region was shorter than the sampling period, the sample
        nearest to it (taken under the same load: warm-up steps precede and the eager profile follows the timed region)."""
        inside = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.06]
        window = "timed region"
        if not inside and self.rows:
            mid = 0.5 * (t0 + t1)
            inside = [min(self.rows, key=lambda tr: abs(tr[0] - mid))[1]]
            window = "nearest sample to the timed region"
        sm, mx, pw, reasons = [], [], [], set()
        for r in inside:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            try:
                pw.append(float(r[2]))
            except (ValueError, IndexError):
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_min_mhz": min(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "window": window, "power_w_max": max(pw) if pw else None}


# =====================================================================================================
# workloads
# =====================================================================================================
def workload_spec(name, world, batch_override=None):
    """-> dict(kind, B (utterances on THIS rank for uniform kinds), T, S, scaling, text)"""
    if name == "c4":
        total = batch_override * world if batch_override else C4_UTTERANCES
        if total % world:
            raise SystemExit(f"bench.py: c4 shards {total} utterances evenly; {world} GPUs do not divide it")
        B = total // world
        return dict(kind="uniform", B=B, T=FRAMES_10S, S=TEXT_LEN, scaling="strong", total=total,
                    text=f"C4: 50-step-style CFG DDPM sampling of {total} x 10 s utterances sharded by utterance over {world} GPU(s) "
                         f"({B} per GPU; T={FRAMES_10S} frames, S={TEXT_LEN} text tokens), repo-default DiT (H=768, L=5, heads=1)")
    if name == "c2":
        B = batch_override or 16
        return dict(kind="uniform", B=B, T=FRAMES_10S, S=TEXT_LEN, scaling="weak", total=B * world,
                    text=f"C2: 50-step-style CFG DDPM sampling, batch {B} x 10 s utterances per GPU (T={FRAMES_10S} frames, "
                         f"S={TEXT_LEN} text tokens), repo-default DiT (H=768, L=5, heads=1)")
    if name == "c3":
        B = batch_override or 4
        return dict(kind="uniform", B=B, T=2250, S=192, scaling="weak", total=B * world,
                    text=f"C3: long-utterance stress, batch {B} x 30 s utterances per GPU (T=2250 frames, S=192 text tokens), "
                         "CFG DDPM sampling, repo-default DiT (H=768, L=5, heads=1)")
    if name == "c5":
        total = batch_override * world if batch_override else C4_UTTERANCES
        return dict(kind="ragged", scaling="strong", total=total,
                    text=f"C5: {total} utterances of 2-20 s (random.seed(0); T_i = 75 s, S_i = round(6.4 s)), each at its own length "
                         f"(packed, unpadded), balanced by forward cost over {world} GPU(s); CFG DDPM sampling, repo-default DiT")
    raise SystemExit(f"bench.py: unknown workload {name}")


def workload_config(args, spec, world, extra=None):
    cfg = {"workload": spec["text"], "name": args.workload, "utterances_total": spec["total"], "guidance_scale": GUIDANCE,
           "diffusion_steps": args.steps, "sharding": f"utterances over {world} GPU(s), no in-step collective",
           "l2": "working set per step (0.7 GB at 16 utterances, 11 GB at 256) exceeds the 126 MB L2; no explicit flush",
           "parity_bar_rel_l2": {"bf16": 2e-2, "fp32": 1e-4}}
    if spec["kind"] == "uniform":
        cfg.update({"batch_per_gpu": spec["B"], "frames": spec["T"], "text_tokens": spec["S"]})
    if extra:
        cfg.update(extra)
    return cfg


# =====================================================================================================
# reference arm / cpu baseline: the reference's own modules (oracle/_ref) or the oracle port, on the host cores
# =====================================================================================================
def cpu_cfg_steps(steps, warmup, max_seconds=None):
    """Times `steps` CFG denoising steps of ONE utterance (B=1, T=750, S=64, fp32) on the CPU: two reference forwards
    (DiTTO.py:66-94) + CFG combine + the update of SpeechGenerator.py:137-147.  -> (done, seconds, cores, kind)"""
    import torch
    from oracle import ditto_oracle as O   # checker / CPU baseline only
    from oracle import ref_loader as R
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = O.OracleConfig(HIDDEN, LAYERS, HEADS, TIME_DIM, HIDDEN, max(steps, 2))
    sd = O.make_state_dict(cfg, 0)
    x, text, _ = O.make_inputs(1, FRAMES_10S, TEXT_LEN, cfg, 1)
    betas, alphas, acp = O.sampler_tables(cfg.diffusion_steps)
    ref, kind = None, "port"
    if R.available():
        try:
            ref, kind = R.build_reference(cfg, sd), "reference"
        except Exception as e:  # noqa: BLE001 -- an import problem on the box must not lose the baseline: fall back to the port
            sys.stderr.write(f"bench.py: oracle/_ref not usable ({e!r}); timing the oracle port instead\n")
    zero_text = torch.zeros_like(text)
    g = torch.Generator().manual_seed(2)
    done, t_total = 0, 0.0
    with torch.no_grad():
        for i in range(warmup + steps):
            t_val = cfg.diffusion_steps - 1 - (i % cfg.diffusion_steps)
            t = torch.full((1,), t_val, dtype=torch.long)
            t0 = time.perf_counter()
            if ref is not None:
                e_c, e_u = ref(x, text, t), ref(x, zero_text, t)
                eps = e_u + GUIDANCE * (e_c - e_u)
            else:
                eps = O.predict_noise(sd, cfg, x, text, t, GUIDANCE)
            z = torch.randn(x.shape, generator=g)
            x = O.p_sample_update(x, eps, z, t, betas, alphas, acp)
            dt = time.perf_counter() - t0
            if i >= warmup:
                done += 1
                t_total += dt
                if max_seconds is not None and t_total > max_seconds:
                    break
            if not torch.isfinite(x).all():  # random-init latents blow up after many steps; restart the state
                x, _, _ = O.make_inputs(1, FRAMES_10S, TEXT_LEN, cfg, 1)
    return done, t_total, cores, kind


def cpu_sample_text(done, cores, kind):
    what = ("the reference's own DiTTO.forward (oracle/_ref: src/model/DiTTO.py + src/components/DiT.py, unmodified)"
            if kind == "reference" else "the CPU oracle port of the reference")
    return (f"{done} CFG denoising steps of ONE utterance of the batch (B=1, T={FRAMES_10S}, S={TEXT_LEN}, fp32; 2 forwards + "
            f"combine + update per step) with {what}, torch CPU, {cores} threads")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    spec = workload_spec(args.workload, max(world, args.gpus, 1), args.batch)
    done, t_total, cores, kind = cpu_cfg_steps(args.steps, args.warmup, max_seconds=150.0)
    ms = t_total / done * 1e3
    value = FRAMES_10S / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "latent frames/sec per denoising step", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": done, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": spec["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, spec, max(world, args.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind, "sample": cpu_sample_text(done, cores, kind)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# =====================================================================================================
# our arm
# =====================================================================================================
class UniformJob:
    """B utterances of T frames / S tokens on this rank: the product's own stepping (one CUDA-graph replay per step)."""

    def __init__(self, torch, D, model, sampler, B, T, S, K, dev, seed):
        self.torch, self.B, self.T, self.S, self.K, self.dev, self.seed = torch, B, T, S, K, dev, seed
        self.sampler = sampler
        g = torch.Generator().manual_seed(seed)
        self.text_host = torch.randn(B, S, HIDDEN, generator=g).pin_memory()
        self.x_host = torch.randn(B, T, HIDDEN, generator=g).pin_memory()
        self.out_host = torch.empty(B, T, HIDDEN).pin_memory()
        self.text = self.text_host.to(dev)
        self.x0 = self.x_host.to(dev)
        self.ctx = sampler._context(self.text, True, None, T)
        self.graph = sampler.step_graph(B, T, S, True, GUIDANCE, self.ctx, True, dev)
        self.frames = B * T
        self.flops_step = 2 * B * forward_flops(T, S)
        self.launches_per_step = self.graph.launches_per_step

    def reset(self):
        self.graph.reset(self.x0, self.K - 1, self.seed)

    def step(self):
        self.graph.replay()

    def result(self):
        return self.graph.x

    def e2e_once(self):
        t_dev = self.text_host.to(self.dev, non_blocking=True)
        x_dev = self.x_host.to(self.dev, non_blocking=True)
        res = self.sampler.sample_latents(t_dev, x_init=x_dev)
        self.out_host.copy_(res, non_blocking=True)

    def e2e_bytes(self):
        return (self.text_host.numel() + self.x_host.numel()) * 4, self.out_host.numel() * 4

    def eager_step(self, state):
        """one un-graphed step through the C-ABI (per-kernel-class profile)"""
        from ditto_tts_b200 import _lib
        from ditto_tts_b200.model import _ptr, _stream
        g = self.graph
        _lib.check(_lib.load().ditto_p_sample_rng(self.sampler.model.engine(), _ptr(g.x), _ptr(g.ctx), _ptr(g.t), _ptr(g.rng), 1,
                                                  GUIDANCE, self.B, self.T, self.S, _ptr(g.eps), _ptr(g.x), _ptr(g.ws), g.ws.numel(),
                                                  1, _stream()), "ditto_p_sample_rng")


class RaggedJob:
    """This rank's cost-balanced share of the C5 utterances, every one at its own length (packed, unpadded)."""

    def __init__(self, torch, D, model, sampler, total, world, rank, K, dev, seed):
        from ditto_tts_b200 import parallel
        from ditto_tts_b200.ragged import RaggedBatch, RaggedStepGraph
        self.torch, self.K, self.dev, self.sampler, self.seed = torch, K, dev, sampler, seed
        T_all, S_all = parallel.c5_lengths(total)
        mine = parallel.balance_by_cost(T_all, world, S_all)[rank]
        self.T = [T_all[i] for i in mine]
        self.S = [S_all[i] for i in mine]
        g = torch.Generator().manual_seed(seed)
        self.text_host = [torch.randn(s, HIDDEN, generator=g).pin_memory() for s in self.S]
        self.texts = [t.to(dev) for t in self.text_host]
        self.rb = RaggedBatch(model, self.texts, self.T, guided=True)
        self.x_host = torch.randn(self.rb.x_rows, HIDDEN, generator=g).pin_memory()
        self.out_host = torch.empty(self.rb.x_rows, HIDDEN).pin_memory()
        self.x0 = self.x_host.to(dev)
        self.graph = RaggedStepGraph(self.rb, GUIDANCE, True)
        self.frames = sum(self.T)
        self.flops_step = sum(2 * forward_flops(t, s) for t, s in zip(self.T, self.S))
        self.launches_per_step = self.graph.launches_per_step
        self.groups = len(self.rb.groups)

    def reset(self):
        self.graph.reset(self.x0, self.K - 1, self.seed)

    def step(self):
        self.graph.replay()

    def result(self):
        return self.graph.x

    def e2e_once(self):
        texts = [t.to(self.dev, non_blocking=True) for t in self.text_host]
        x_dev = self.x_host.to(self.dev, non_blocking=True)
        # per-utterance latents in utterance order, as the public API takes them
        xs = [x_dev[self.rb.x_offset[i]:self.rb.x_offset[i] + self.T[i]] for i in range(len(self.T))]
        res = self.sampler.sample_latents_ragged(texts, self.T, x_init=xs)
        for i, r in enumerate(res):
            o = self.rb.x_offset[i]
            self.out_host[o:o + self.T[i]].copy_(r, non_blocking=True)

    def e2e_bytes(self):
        return (sum(t.numel() for t in self.text_host) + self.x_host.numel()) * 4, self.out_host.numel() * 4

    def eager_step(self, state):
        from ditto_tts_b200 import _lib
        from ditto_tts_b200.model import _ptr, _stream
        g, b = self.graph, self.rb
        _lib.check(_lib.load().ditto_p_sample_ragged_rng(b.model.engine(), _ptr(g.x), b.c_groups, len(b.groups), _ptr(g.t), _ptr(g.rng), 1,
                                                         GUIDANCE, _ptr(g.eps), _ptr(g.x), _ptr(g.ws), g.ws.numel(), 1, _stream()),
                   "ditto_p_sample_ragged_rng")


def timed_job(torch, job, K, W, barrier):
    """W warm-up steps (a fresh job every K steps, so that t never runs below 0), then one K-step job between two CUDA
    events: -> (ms, wall t0, wall t1)."""
    for i in range(W):
        if i % K == 0:
            job.reset()
        job.step()
    job.reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.perf_counter()
    e0.record()
    for _ in range(K):
        job.step()
    e1.record()
    barrier()
    t_wall1 = time.perf_counter()
    return e0.elapsed_time(e1), t_wall0, t_wall1


def dump_outputs(out_dir, x):
    """DIR/latents.npy: the latents `x` as float32 rows [frames, H]; above DUMP_ROWS frames, a fixed seeded sample of
    DUMP_ROWS of them in frame order (the same frames on every run).  -> what the JSON line reports about the dump."""
    import numpy as np
    import torch
    rows = x.detach().reshape(-1, x.shape[-1]).float().cpu()
    n = rows.shape[0]
    if n > DUMP_ROWS:
        rows = rows[torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "latents.npy"), rows.numpy())
    return {"dir": out_dir, "latents": list(rows.shape), "frames_total": n}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import ditto_tts_b200 as D
    from ditto_tts_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    K, W = args.steps, args.warmup
    spec = workload_spec(args.workload, world, args.batch)
    clocks = ClockSampler(local).start()
    torch.manual_seed(0)  # random-init weights of the named architecture (default torch initialisers)
    model = D.DiTTO(hidden_dim=HIDDEN, num_layers=LAYERS, num_heads=HEADS, time_dim=TIME_DIM, text_dim=HIDDEN,
                    diffusion_steps=K, precision=args.precision).to(dev)
    sampler = D.DiTTOSampler(model, guidance_scale=GUIDANCE)
    if spec["kind"] == "uniform":
        job = UniformJob(torch, D, model, sampler, spec["B"], spec["T"], spec["S"], K, dev, 1 + rank)
    else:
        job = RaggedJob(torch, D, model, sampler, spec["total"], world, rank, K, dev, 1 + rank)

    # ---------------- device-resident loop (metric `value`) ----------------
    ms_total, t_wall0, t_wall1 = timed_job(torch, job, K, W, barrier)
    finite = bool(torch.isfinite(job.result()).all())
    dumped = dump_outputs(args.dump_outputs, job.result()) if args.dump_outputs and rank == 0 else None
    clock_summary = clocks.summary(t_wall0, t_wall1)

    # ---------------- end to end through the public API, host buffers ----------------
    job.e2e_once()  # warm (allocations / graph of the public path)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    job.e2e_once()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    # ---------------- per-kernel-class timing (CUDA events on the launching stream, eager steps) ----------------
    # The profiled steps must see the clock the timed region saw: ~1.2 s of back-to-back graph replays first (the SM clock
    # sags to the power-capped level again after the host-side pause of the e2e copy), then the eager steps with no gap;
    # the clock samples of exactly that window choose the roofline denominator.
    ms_step_est = ms_total / K
    job.reset()
    for i in range(max(1, min(5000, int(1200.0 / max(ms_step_est, 1e-3))))):
        if i % K == 0:
            job.reset()
        job.step()
    job.reset()
    torch.cuda.synchronize()
    t_prof0 = time.perf_counter()
    _lib.profile_start()
    prof_steps = min(K, 5)
    for i in range(prof_steps):
        job.eager_step(i)
    prof = _lib.profile_stop()
    torch.cuda.synchronize()
    t_prof1 = time.perf_counter()
    prof_clocks = clocks.summary(t_prof0, t_prof1)

    # ---------------- C2 beside C4 on one GPU (BASELINE configs[1]; continuity with round 1) ----------------
    c2 = None
    if world == 1 and args.workload == "c4" and not args.no_c2:
        job2 = UniformJob(torch, D, model, sampler, 16, FRAMES_10S, TEXT_LEN, K, dev, 101)
        ms2, w0, w1 = timed_job(torch, job2, K, W, barrier)
        ck2 = clocks.summary(w0, w1)
        ms2_step = ms2 / K
        job2.e2e_once()
        barrier()
        f0.record()
        job2.e2e_once()
        f1.record()
        barrier()
        c2 = {"workload": workload_spec("c2", 1)["text"], "value": job2.frames / (ms2_step / 1e3), "unit": "frames/s",
              "ms_per_step": ms2_step, "timed_ms": ms2,
              "algorithmic_tflops": job2.flops_step / (ms2_step / 1e3) / 1e12,
              "e2e_value": job2.frames * K / (f0.elapsed_time(f1) / 1e3),
              "rtf_10s_utterance_batch_latency": ms2_step * K / 1e3 / 10.0,
              "clocks": {k: ck2.get(k) for k in ("sm_mhz", "sm_max_mhz", "samples", "reasons")}}
        del job2
    # ---------------- one 10 s utterance alone (the metric's RTF half: latency of a single request) ----------------
    single = None
    if world == 1 and args.workload == "c4" and not args.no_c2:
        job1 = UniformJob(torch, D, model, sampler, 1, FRAMES_10S, TEXT_LEN, K, dev, 201)
        ms1_job, _, _ = timed_job(torch, job1, K, W, barrier)
        job1.e2e_once()
        barrier()
        f0.record()
        job1.e2e_once()
        f1.record()
        barrier()
        single = {"workload": f"one 10 s utterance (B=1, T={FRAMES_10S}, S={TEXT_LEN}), {K}-step CFG sampling", "job_latency_ms": ms1_job,
                  "rtf": ms1_job / 1e3 / 10.0, "ms_per_step": ms1_job / K,
                  "e2e_latency_ms": f0.elapsed_time(f1), "e2e_rtf": f0.elapsed_time(f1) / 1e3 / 10.0,
                  "launches_per_step": int(job1.launches_per_step)}
        del job1
    clocks.stop()

    # ---------------- reduce over ranks: time = max, frames / flops = sum ----------------
    red_max = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    red_sum = torch.tensor([float(job.frames), float(job.flops_step)], dtype=torch.float64, device=dev)
    gather_ms = 0.0
    if world > 1:
        dist.all_reduce(red_max, op=dist.ReduceOp.MAX)
        dist.all_reduce(red_sum, op=dist.ReduceOp.SUM)
        if spec["kind"] == "uniform":
            # NCCL is used only to gather the outputs (SURVEY.md 8e); timed separately from the step metric
            xa = job.result()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            gathered = torch.empty((world * xa.shape[0],) + tuple(xa.shape[1:]), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(gathered, xa)
            barrier()
            g0.record()
            dist.all_gather_into_tensor(gathered, xa)
            g1.record()
            barrier()
            gather_ms = g0.elapsed_time(g1)
    ms_total, ms_e2e = float(red_max[0]), float(red_max[1])
    frames_all, flops_all = float(red_sum[0]), float(red_sum[1])

    if rank == 0:
        peaks = load_peaks()
        ms_step = ms_total / K
        value = frames_all / (ms_step / 1e3)
        peak_kind, peak = choose_peak(peaks, prof_clocks if prof_clocks.get("sm_mhz") else clock_summary)
        tot_prof_ms = sum(v["ms"] for v in prof.values()) or 1.0
        dom_name = max(prof, key=lambda k_: prof[k_]["ms"])
        dom = prof[dom_name]
        tc_ms = sum(v["ms"] for k_, v in prof.items() if k_.startswith("tc_gemm"))
        tc_flops = sum(v["flops"] for k_, v in prof.items() if k_.startswith("tc_gemm"))
        ach = dom["flops"] / (dom["ms"] / 1e3) / 1e12 if dom["flops"] else 0.0
        traffic, traffic_src = traffic_for(dom_name)
        step_tflops_gpu = (flops_all / world) / (ms_step / 1e3) / 1e12     # per GPU
        roofline = {"kernel": dom_name, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    "frac_burst": ach / peaks["burst"], "frac_sustained": ach / peaks["sustained"],
                    "peak_source": f"{peaks['source']}, {peak_kind} (median SM clock {prof_clocks.get('sm_mhz')} MHz over "
                                   f"{prof_clocks.get('samples')} samples of the profiled steps, {clock_summary.get('sm_mhz')} of "
                                   f"{clock_summary.get('sm_max_mhz')} MHz in the timed region)",
                    "traffic": traffic, "traffic_source": traffic_src,
                    "launch_us": dom["ms"] / dom["launches"] * 1e3, "flops_per_launch": dom["flops"] / dom["launches"],
                    "share_of_step": dom["ms"] / tot_prof_ms,
                    "timing": f"CUDA events around every launch of {prof_steps} eager steps on rank 0, run back to back behind "
                              f"~1.2 s of graph replays (same sustained clock as the timed region)",
                    "profiled_clocks": {k_: prof_clocks.get(k_) for k_ in ("sm_mhz", "sm_min_mhz", "samples", "window")},
                    "profiled_step_ms": tot_prof_ms / prof_steps,
                    "tc_gemm_family": {"achieved": tc_flops / (tc_ms / 1e3) / 1e12 if tc_ms else 0.0,
                                       "share_of_step": tc_ms / tot_prof_ms},
                    "whole_step": {"algorithmic_tflops_per_gpu": step_tflops_gpu, "frac_of_peak": step_tflops_gpu / peak,
                                   "frac_of_burst": step_tflops_gpu / peaks["burst"],
                                   "frac_of_sustained": step_tflops_gpu / peaks["sustained"]},
                    "per_class_ms_per_step": {k_: round(v["ms"] / prof_steps, 4) for k_, v in sorted(prof.items())},
                    "per_class": per_class_roofline(prof, peak, peaks["hbm"]),
                    "per_class_launches_per_step": {k_: v["launches"] // prof_steps for k_, v in sorted(prof.items())}}
        cpu = None
        if world == 1:
            done, t_cpu, cores, kind = cpu_cfg_steps(steps=12, warmup=1, max_seconds=12.0)
            cpu = {"value": FRAMES_10S / (t_cpu / done), "unit": "frames/s", "cores": cores, "kind": kind,
                   "sample": cpu_sample_text(done, cores, kind)}
        h2d, d2h = job.e2e_bytes()
        extra = {"length_groups_rank0": job.groups, "valid_frames_total": frames_all} if spec["kind"] == "ragged" else None
        line = {
            "metric": "latent frames/sec per denoising step", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": W, "timed_ms": ms_total, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": spec["scaling"], "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
            "config": workload_config(args, spec, world, extra),
            "rtf": {"job_latency_s": ms_step * K / 1e3, "rtf_10s_utterance": ms_step * K / 1e3 / 10.0,
                    "rtf_per_audio_second": ms_step * K / 1e3 / (frames_all / 75.0)},
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": {"value": frames_all * K / (ms_e2e / 1e3), "unit": "frames/s", "h2d_bytes_per_step": h2d / K,
                    "d2h_bytes_per_step": d2h / K, "ms_total": ms_e2e,
                    "api": "DiTTOSampler.sample_latents(text_emb, x_init) from pinned host tensors, final latents to host; one K-step job"},
            "gpu_launches": int(job.launches_per_step * K), "launches_per_step": int(job.launches_per_step),
            "stepping": "cuda-graph replay per step (libditto_b200 kernels only)", "clocks": clock_summary,
            "outputs_finite": finite, "output_gather_ms": gather_ms,
        }
        if c2 is not None:
            line["c2"] = c2
        if single is not None:
            line["rtf"]["single_utterance"] = single
        if dumped is not None:
            line["dump_outputs"] = dumped
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=["c2", "c3", "c4", "c5"], default="c4")
    ap.add_argument("--batch", type=int, default=None, help="utterances per GPU (overrides the workload's count)")
    ap.add_argument("--precision", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--no-c2", action="store_true", help="skip the C2 side measurement of the single-GPU c4 run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the final latents of the timed job to DIR/latents.npy (float32, at most DUMP_ROWS frames)")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("bench.py: --steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if args.gpus > 1 and world == 1:
            # convenience: re-launch under torchrun
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                   "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), __file__,
                   "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup),
                   "--workload", args.workload, "--precision", args.precision]
            if args.batch:
                cmd += ["--batch", str(args.batch)]
            if args.dump_outputs:
                cmd += ["--dump-outputs", args.dump_outputs]
            raise SystemExit(subprocess.call(cmd))
        run_ours(args)


if __name__ == "__main__":
    main()
