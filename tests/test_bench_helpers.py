"""bench.py's host-side helpers (no GPU): the nvidia-smi clock parser, the cpu_baseline leg and the CLI contract."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
bench = importlib.util.module_from_spec(spec)
spec.loader.exec_module(bench)


def test_clock_sampler_parses_nvidia_smi_rows_and_flags_throttling():
    s = bench.ClockSampler(0)

    class _P:  # a finished process
        def terminate(self): pass
        def wait(self, timeout=None): return 0
        def kill(self): pass

    s.proc = _P()
    s.rows = ["0, 1965, 1965, 701.7, Not Active, Not Active, Not Active, Not Active",
              "0, 1950, 1965, 998.2, Not Active, Not Active, Not Active, Active",
              "0, 1200, 1965, 640.0, Not Active, Active, Not Active, Not Active", "garbage"]
    out = s.stop()
    assert out["sm_mhz"] == 1950.0 and out["sm_max_mhz"] == 1965.0 and out["samples"] == 3
    assert out["reasons"] == ["hw_thermal_slowdown", "sw_power_cap"] and out["power_w_max"] == 998.2
    assert bench.ClockSampler(0).stop()["reasons"] == ["nvidia-smi unavailable"]


def test_cpu_baseline_runs_the_oracle_on_a_bounded_sample(monkeypatch):
    import time as _t

    ticks = iter(range(0, 10_000, 6))  # pretend every timing call is 6 s apart: one pass, then the 10 s budget is spent
    monkeypatch.setattr(bench.time, "perf_counter", lambda: float(next(ticks)))
    out = bench.cpu_baseline(world=2, batch=256, bucket_numels=[1000, 2048, 77])
    assert out["kind"] == "port" and out["cores"] == 1 and out["value"] > 0 and "oracle/allreduce_oracle.c" in out["sample"]
    assert "x 2 ranks" in out["sample"] and out["host_cpus"] == os.cpu_count()


def test_cli_contract_and_no_cpu_fallback():
    help_text = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120).stdout
    for flag in ("--gpus", "--steps", "--warmup", "--impl"):
        assert flag in help_text
    # without a GPU the product arm must refuse to run rather than fall back to a CPU path (devices hidden, so this holds on GPU hosts too)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                         timeout=300, env=env)
    assert res.returncode != 0 and "no CPU fallback" in (res.stderr + res.stdout)
    assert not any(line.strip().startswith("{") for line in res.stdout.splitlines())


def test_dump_outputs_writes_float32_files_with_a_fixed_sample(tmp_path):
    """--dump-outputs on CPU tensors: four float32 files; arrays over max_elems become the elements at the same sorted,
    seeded positions in every run; at the default size the four files stay well under 64 MB."""
    import types

    import numpy as np
    import torch

    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(64, 48), torch.nn.ReLU(), torch.nn.Linear(48, 10))
    x, y = torch.randn(32, 64), torch.randint(0, 10, (32,))
    logits = model(x)
    loss = torch.nn.functional.cross_entropy(logits, y)
    loss.backward()
    tr = types.SimpleNamespace(torch=torch, ddp=model, last_loss=loss.detach(), last_logits=logits.detach())
    params = [p for p in model.parameters()]
    n = sum(p.numel() for p in params)  # 3600: sampled at max_elems=1000, written whole at the default
    grads = torch.cat([p.grad.reshape(-1) for p in params]).numpy()

    for run in ("a", "b"):
        bench.Trainer.dump_outputs(tr, str(tmp_path / run), max_elems=1000)
    bench.Trainer.dump_outputs(tr, str(tmp_path / "full"))
    assert sorted(os.listdir(tmp_path / "a")) == ["grads.npy", "logits.npy", "loss.npy", "params.npy"]
    got = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["loss.npy"].tolist() == [loss.item()] and got["logits.npy"].size == 320  # small arrays whole
    assert got["grads.npy"].size == got["params.npy"].size == 1000
    for f, a in got.items():
        assert np.array_equal(a, np.load(tmp_path / "b" / f)), f  # same positions in every run
    idx = np.sort(np.random.default_rng(n).choice(n, size=1000, replace=False))
    assert np.array_equal(got["grads.npy"], grads[idx]) and np.array_equal(np.load(tmp_path / "full" / "grads.npy"), grads)
    max_elems = bench.Trainer.dump_outputs.__defaults__[0]
    assert max_elems == 1 << 21 and 4 * max_elems * 4 <= 64 << 20  # four float32 files of at most max_elems each


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert res.returncode == 2 and "--steps must be at least 1" in res.stderr
