"""bench.py's algorithmic-work formulas (the numerators of every roofline fraction it reports) against the figures in
BASELINE.md section 3 / SURVEY.md section 8(d), and the shape of the reference-arm JSON line.  CPU only."""
import importlib.util
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("vcla_bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_algorithmic_work_matches_baseline_tables(bench):
    # BASELINE.md: config 2 (B=8, S=128, N=256): prefill 14.73 TFLOP, decode 3 682 GB over 255 steps
    assert bench.prefill_flops(8, 128) == pytest.approx(14.73e12, rel=5e-3)
    dec = sum(bench.decode_step_bytes(8, 128 + i) for i in range(255))
    assert dec == pytest.approx(3682e9, rel=5e-3)
    # config 3 (B=32, S=192): prefill 85.64 TFLOP, decode 4 780 GB
    assert bench.prefill_flops(32, 192) == pytest.approx(85.64e12, rel=5e-3)
    assert sum(bench.decode_step_bytes(32, 192 + i) for i in range(255)) == pytest.approx(4780e9, rel=5e-3)
    # config 5 (B=16, S=1088, N=512): prefill 233.3 TFLOP, decode 12 593 GB
    assert bench.prefill_flops(16, 1088) == pytest.approx(233.3e12, rel=1e-2)
    assert sum(bench.decode_step_bytes(16, 1088 + i) for i in range(511)) == pytest.approx(12593e9, rel=5e-3)
    # per-step weight bytes: 13.361 GB (SURVEY 8d)
    assert bench.decode_step_bytes(0, 0) == pytest.approx(13.361e9, rel=1e-3)


def test_synthetic_inputs_follow_survey_8d(bench):
    px, ids = bench.synth_inputs(4, T=64)
    assert tuple(px.shape) == (4, 3, 224, 224) and tuple(ids.shape) == (4, 64)
    assert ids[:, 0].tolist() == [1] * 4 and ids[:, 1].tolist() == [49954] * 4 and ids[:, 2].tolist() == [49955] * 4
    assert int(ids[:, 3:].min()) >= 3 and int(ids[:, 3:].max()) < 49954


def test_native_arm_refuses_to_run_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("has a GPU")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_dump_outputs_and_its_arguments(bench, tmp_path, monkeypatch):
    """--dump-outputs DIR writes the timed step's tokens exactly (float64) as DIR/tokens.npy; --steps below 1 is refused, and so is
    --dump-outputs with any arm but the native one, before any work starts."""
    import numpy as np
    import torch
    tok = torch.randint(0, 49958, (8, 256), generator=torch.Generator().manual_seed(0))
    bench.dump_outputs(str(tmp_path / "out"), tok)
    got = np.load(tmp_path / "out" / "tokens.npy")
    assert got.dtype == np.float64 and got.shape == (8, 256) and np.array_equal(got, tok.numpy())
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "3", "--dump-outputs", str(tmp_path)])
    assert bench.parse().steps == 3
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)], ["--impl", "hf-cuda", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            bench.parse()


def test_native_arm_times_steps_and_dumps_that_runs_tokens(bench, tmp_path, monkeypatch, capsys):
    """run_native hands --steps and --warmup to the timed configuration and dumps the tokens that timed run returned (the device stands
    in as a fake run_config: no GPU here)."""
    import numpy as np
    import torch
    from visualcla import _native
    for k in ("WORLD_SIZE", "RANK", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: None)
    monkeypatch.setattr(_native, "load", lambda: type("Lib", (), {"vcla_set_pdl": staticmethod(lambda on: None)})())
    tok = torch.randint(0, 49958, (8, 256), generator=torch.Generator().manual_seed(1))
    calls = []

    def fake_run_config(args, world, rank, Bl, T, n_new, steps, warmup, with_e2e, with_trace):
        calls.append((Bl, T, n_new, steps, warmup, with_e2e, with_trace))
        return {"value": 1.0, "ms": 750.0 * steps, "steps": steps, "launches": 0, "clocks": {}, "e2e": {}, "tokens": tok}

    monkeypatch.setattr(bench, "run_config", fake_run_config)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "4", "--warmup", "2", "--no-extras", "--no-cpu-baseline",
                                      "--dump-outputs", str(tmp_path / "dump")])
    bench.run_native(bench.parse())
    assert calls == [(8, 64, 256, 4, 2, True, True)]
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == 4 and line["ms_per_step"] == pytest.approx(750.0)
    assert np.array_equal(np.load(tmp_path / "dump" / "tokens.npy"), tok.numpy())


def test_hf_cuda_arm_times_exactly_steps(bench, monkeypatch):
    """The informational HF arm times --steps generations after --warmup ones (at least one, to check the output shape)."""
    import argparse
    import torch
    monkeypatch.delenv("RANK", raising=False)
    calls = []

    def fake_step_builder(B, T, n_new, dt):
        def step():
            calls.append(1)
            return torch.zeros(B, n_new, dtype=torch.long)
        return step

    class FakeEvent:
        def __init__(self, **k):
            pass

        def record(self):
            pass

        def elapsed_time(self, other):
            return 700.0

    monkeypatch.setattr(bench, "hf_cuda_step", fake_step_builder)
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    for f in ("set_device", "synchronize", "empty_cache"):
        monkeypatch.setattr(torch.cuda, f, lambda *a: None)
    for warmup, steps in ((2, 7), (0, 1), (5, 5)):
        calls.clear()
        ns = argparse.Namespace(hf_dtype="float16", batch_per_gpu=2, new_tokens=3, prompt_tokens=4, warmup=warmup, steps=steps)
        line = bench.run_hf_cuda(ns, emit=False)
        assert len(calls) == max(1, warmup) + steps
        assert line["steps"] == steps and line["warmup"] == max(1, warmup) and line["ms_per_step"] == pytest.approx(700.0 / steps)
    calls.clear()
    assert bench.hf_cuda_sample(2, 4, 3, steps=2)["steps"] == 2 and len(calls) == 3     # the bounded block of the default native line


def test_insitu_trace_labelling_and_durations(bench, monkeypatch):
    """bench.py's in-situ roofline: kernels of one graph-replayed decode step are labelled by order (per layer qkv, o, gate/up, down; the
    129th swap-AB GEMM is lm_head) and a kernel's duration is its successor's dependency-resolved time minus its own, so the
    durations add up to the step."""
    import torch

    class FakeEngine:
        def __init__(self):
            self.enabled = False

        def decode_step(self, *a, **k):
            pass

        def trace_enable(self, n):
            self.enabled = n > 0

        def trace_read(self):
            # (tag, t_entry, t_dep, t_exit) in ns; cluster split-K schedule: embed, 32 x [qkv, attn, o, gate_up, down], lm_head, logits1, logits2, advance
            t, ev = 1000, [(13, 900, 1000, 0)]
            per = {"qkv": 17500, "attn": 11000, "o": 10500, "gu": 29500, "d": 19000}
            for _ in range(32):
                for tag, key in ((1, "qkv"), (4, "attn"), (1, "o"), (1, "gu"), (1, "d")):
                    t += {13: 2500}.get(ev[-1][0], 0) if len(ev) == 1 else 0
                    ev.append((tag, t - 5000, t, t + 100))
                    t += per[key]
            for tag, dur in ((1, 61000), (10, 4600), (11, 1600), (12, 2000)):
                ev.append((tag, t - 1000, t, 0))
                t += dur
            return ev

    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    mean, count, total = bench.insitu_decode_kernels(FakeEngine(), None)
    assert count["qkv"] == 32 and count["o_proj"] == 32 and count["gate_up"] == 32 and count["down_proj"] == 32 and count["lm_head"] == 1
    assert mean["gate_up"] == pytest.approx(29.5) and mean["qkv"] == pytest.approx(17.5) and mean["down_proj"] == pytest.approx(19.0)
    assert mean["lm_head"] == pytest.approx(61.0) and mean["attn_decode"] == pytest.approx(11.0)
    assert total == pytest.approx(sum(mean[k] * count[k] for k in mean), rel=1e-6)
    assert bench.GEMM_BYTES["gate_up"] == 2 * 11008 * 4096 * 2 and bench.GEMM_BYTES["lm_head"] == 49958 * 4096 * 2
