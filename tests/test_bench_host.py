"""Host-side pieces of bench.py that run without a GPU: the work model, the clock-sample window, the timed-step count
and the output dump."""
import importlib.util
import json
import os
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
bench = importlib.util.module_from_spec(spec)
spec.loader.exec_module(bench)


def test_flop_model_matches_survey_numbers():
    """SURVEY.md 8d: 86.35 GFLOP per sequence per forward at T = 750, S = 64 (repo-default model)."""
    assert abs(bench.forward_flops(750, 64) / 1e9 - 86.35) < 0.01
    assert abs(bench.forward_flops(2250, 192) / 1e9 - 315.3) < 0.1


def test_clock_sampler_keeps_samples_of_the_timed_region():
    s = bench.ClockSampler(0)
    row = lambda mhz, cap: [str(mhz), "1965", "700.0", "Not Active", "Not Active", "Not Active", "Active" if cap else "Not Active"]
    s.rows = [(9.90, row(1965, False)), (10.02, row(1850, True)), (10.07, row(1800, True)), (10.12, row(1840, False)),
              (10.40, row(1965, False))]
    out = s.summary(10.0, 10.15)
    assert out["samples"] == 3 and out["sm_mhz"] == 1840.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"] and out["window"] == "timed region"
    # a region shorter than the sampling period falls back to the nearest sample and says so
    out = s.summary(10.20, 10.22)
    assert out["samples"] == 1 and out["window"].startswith("nearest")
    s.rows = []
    assert s.summary(0.0, 1.0)["samples"] == 0


def test_peak_choice_follows_the_sampled_clock():
    peaks = dict(burst=1674.1, sustained=1428.7, hbm=6554.6, source="t")
    assert bench.choose_peak(peaks, {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0}) == ("burst", 1674.1)
    assert bench.choose_peak(peaks, {"sm_mhz": 1400.0, "sm_max_mhz": 1965.0}) == ("sustained", 1428.7)
    assert bench.choose_peak(peaks, {"sm_mhz": None, "sm_max_mhz": None})[0] == "burst"   # no sample: the stricter denominator


def test_workloads_follow_baseline_configs():
    """BASELINE.json configs[3]: 256 utterances sharded 256 / N (strong scaling); configs[1]: 16 per GPU; configs[2]: 4 x 30 s."""
    for n in (1, 2, 4, 8):
        w = bench.workload_spec("c4", n)
        assert w["B"] * n == 256 and w["scaling"] == "strong" and (w["T"], w["S"]) == (750, 64)
    assert bench.workload_spec("c2", 8)["B"] == 16 and bench.workload_spec("c2", 8)["scaling"] == "weak"
    w = bench.workload_spec("c3", 1)
    assert (w["B"], w["T"], w["S"]) == (4, 2250, 192)
    assert bench.workload_spec("c5", 8)["kind"] == "ragged"
    # the default (what the driver runs) is C4
    import argparse
    assert "c4" in open(os.path.join(ROOT, "bench.py")).read().split('"--workload"')[1].split(")")[0]


def test_traffic_is_reported_only_for_the_source_it_was_captured_from(tmp_path, monkeypatch):
    sha = bench.csrc_sha()
    assert len(sha) == 16
    prof = tmp_path / "profiles"
    prof.mkdir()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    monkeypatch.setattr(bench, "csrc_sha", lambda: sha)
    (prof / "traffic.json").write_text(json.dumps({"_csrc_sha": "stale", "tc_gemm.glu": 1.5e8}))
    assert bench.traffic_for("tc_gemm.glu")[0] is None
    (prof / "traffic.json").write_text(json.dumps({"_csrc_sha": sha, "tc_gemm.glu": 1.5e8}))
    assert bench.traffic_for("tc_gemm.glu")[0] == 1.5e8


def test_traffic_file_names_known_profile_classes():
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
        t = json.load(f)
    keys = [k for k in t if not k.startswith("_")]
    assert "tc_gemm.glu" in keys                       # the dominant kernel of the bench line
    assert all(isinstance(t[k], float) and t[k] > 0 for k in keys)


def test_per_class_roofline_picks_the_longer_bound():
    """A GEMM class is held to the tensor peak, a streaming class to the HBM copy peak; frac = roofline time / measured time."""
    prof = {"tc_gemm.glu": {"ms": 2.0, "flops": 2.0e12, "bytes": 1.0e9, "launches": 1},      # 2 TFLOP in 2 ms = 1000 TFLOP/s
            "adaln_ln": {"ms": 1.0, "flops": 0.0, "bytes": 5.0e9, "launches": 1},            # 5 GB in 1 ms = 5000 GB/s
            "idle": {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0}}
    out = bench.per_class_roofline(prof, 1400.0, 6500.0)
    assert "idle" not in out
    assert out["tc_gemm.glu"]["bound"] == "tensor" and out["tc_gemm.glu"]["unit"] == "TFLOP/s"
    assert abs(out["tc_gemm.glu"]["achieved"] - 1000.0) < 1e-6 and abs(out["tc_gemm.glu"]["frac"] - 1000.0 / 1400.0) < 1e-3
    assert out["adaln_ln"]["bound"] == "hbm" and abs(out["adaln_ln"]["frac"] - 5000.0 / 6500.0) < 1e-3
    assert all(0.0 < v["frac"] <= 1.0 for v in out.values())


def test_timed_region_is_exactly_steps_of_one_job():
    """--steps K: K steps between the two CUDA events, after the W warm-up steps; no step runs past t = 0."""
    log = []

    class Event:
        def __init__(self, enable_timing):
            pass

        def record(self):
            log.append("event")

        def elapsed_time(self, other):
            return 12.5

    class Job:
        def __init__(self, K):
            self.K, self.t = K, None

        def reset(self):
            self.t = self.K - 1

        def step(self):
            assert self.t is not None and self.t >= 0
            self.t -= 1
            log.append("step")

    fake_torch = types.SimpleNamespace(cuda=types.SimpleNamespace(Event=Event))
    for K, W in ((7, 3), (2, 5), (50, 0), (1, 1)):
        log.clear()
        ms, t0, t1 = bench.timed_job(fake_torch, Job(K), K, W, lambda: None)
        assert ms == 12.5 and t0 <= t1
        assert log.count("event") == 2 and log.count("step") == W + K
        first = log.index("event")
        assert log[first + 1:] == ["step"] * K + ["event"]


def test_dump_outputs_writes_float32_latents_within_budget(tmp_path):
    """Small outputs are written whole; large ones as the same seeded sample of frames on every call, under 64 MB."""
    x = torch.randn(2, 5, 768)
    info = bench.dump_outputs(str(tmp_path / "small"), x)
    got = np.load(tmp_path / "small" / "latents.npy")
    assert got.dtype == np.float32 and np.array_equal(got, x.reshape(-1, 768).numpy())
    assert info["latents"] == [10, 768] and info["frames_total"] == 10
    big = torch.randn(3, 6000, 768)
    bench.dump_outputs(str(tmp_path / "a"), big)
    bench.dump_outputs(str(tmp_path / "b"), big)
    a, b = np.load(tmp_path / "a" / "latents.npy"), np.load(tmp_path / "b" / "latents.npy")
    assert a.shape == (bench.DUMP_ROWS, 768) and np.array_equal(a, b)
    assert os.path.getsize(tmp_path / "a" / "latents.npy") < 64e6
    rows = big.reshape(-1, 768).numpy()
    idx = [int(np.flatnonzero((rows == r).all(1))[0]) for r in a[:50]]
    assert idx == sorted(idx)                                   # frames kept in frame order
