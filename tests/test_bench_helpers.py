"""Host-side helpers of bench.py / tools (no GPU needed), and one end-to-end `bench.py --dump-outputs` run on the GPU."""
import importlib.util
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_clock_sampler_parsing():
    bench = _load(os.path.join(ROOT, "bench.py"), "bench_mod")
    s = bench.ClockSampler(2)
    s.proc = type("P", (), {"terminate": lambda self: None, "wait": lambda self, timeout=None: 0, "kill": lambda self: None})()
    s.t_mark = 100.0
    s.lines = [(101.0 + i, ln) for i, ln in enumerate([
        "0, 1965, 1965, 512.3, Not Active, Not Active, Not Active, Active",
        "1, 1800, 1965, 700.0, Not Active, Not Active, Not Active, Not Active",
        "2, 300, 1965, 90.0, Active, Not Active, Not Active, Not Active",      # GPU outside the job: ignored
        "garbage line",
        "0, 1900, 1965, 650.0, Not Active, Not Active, Not Active, Active",
    ])]
    s.lines.insert(0, (50.0, "0, 400, 1965, 90.0, Not Active, Not Active, Not Active, Not Active"))   # before the timed region: ignored
    out = s.stop()
    assert out["sm_mhz"] == 1900 and out["sm_max_mhz"] == 1965 and out["samples"] == 3
    assert out["reasons"] == ["sw_power_cap"] and out["power_w_max"] == 700.0 and out["scope"] == "timed region"
    # a timed region too short to be sampled (8 GPUs, ~0.2 s): the loaded warm-up samples are reported instead of `null`
    s2 = bench.ClockSampler(2)
    s2.proc = s.proc
    s2.t_mark = 200.0
    s2.lines = [(150.0, "0, 1700, 1965, 800.0, Not Active, Not Active, Not Active, Active"),
                (150.1, "1, 1710, 1965, 810.0, Not Active, Not Active, Not Active, Active")]
    out2 = s2.stop()
    assert out2 is not None and out2["samples"] == 2 and out2["scope"] == "warm-up + timed region"


def test_model_kwargs_and_metric_config():
    bench = _load(os.path.join(ROOT, "bench.py"), "bench_mod2")
    kw = bench.model_kwargs("llama125m")
    assert kw["vocab_size"] == 50257 and kw["hidden_size"] == 768 and kw["num_key_value_heads"] == 12
    assert "tokens/sec" in bench.METRIC


def test_reference_arm_reports_unavailable_instead_of_crashing(monkeypatch, capsys):
    """Without a GPU (or without the install) `--impl reference` must print a JSON line and exit 0."""
    bench = _load(os.path.join(ROOT, "bench.py"), "bench_mod3")
    args = type("A", (), dict(steps=2, warmup=1, model="llama125m", batch=2, seq=16, n_acc=1))()
    out = bench.run_reference_arm(args)
    assert out["impl"] == "reference"
    assert "unavailable" in out or "value" in out


def test_dump_outputs_writes_loss_and_sampled_params(tmp_path, monkeypatch):
    """`bench.py --dump-outputs DIR`: float32 loss and weights; a vector above the cap is sampled the same way on every call."""
    import numpy as np
    import torch
    bench = _load(os.path.join(ROOT, "bench.py"), "bench_mod4")
    monkeypatch.setattr(bench, "DUMP_PARAM_SAMPLE", 1000)
    sched = type("S", (), dict(count_grad_tot=7))()
    small = type("T", (), dict(params=torch.randn(1000).bfloat16(), loss_host=torch.tensor([2.5]), micro_batches=9, sched=sched))()
    bench.dump_outputs(str(tmp_path / "small"), small)
    loss, params = np.load(tmp_path / "small" / "loss.npy"), np.load(tmp_path / "small" / "params.npy")
    assert loss.dtype == np.float32 and loss.tolist() == [2.5]
    assert params.dtype == np.float32 and np.array_equal(params, small.params.float().numpy())
    for name, want in (("micro_batches", 9), ("count_grad_tot", 7)):        # whether two dumps took the same schedule
        got = np.load(tmp_path / "small" / f"{name}.npy")
        assert got.dtype == np.float64 and got.tolist() == [want]
    big = type("T", (), dict(params=torch.arange(5000, dtype=torch.float32), loss_host=torch.tensor([1.0]), micro_batches=9, sched=sched))()
    bench.dump_outputs(str(tmp_path / "a"), big)
    bench.dump_outputs(str(tmp_path / "b"), big)
    a, b = np.load(tmp_path / "a" / "params.npy"), np.load(tmp_path / "b" / "params.npy")
    assert a.shape == (1000,) and np.array_equal(a, b)
    assert np.all(np.diff(a) >= 0) and a.min() >= 0 and a.max() < 5000     # sorted indices into the vector


@pytest.mark.gpu
def test_bench_dump_outputs_on_the_gpu(tmp_path):
    """`bench.py --steps 1 --dump-outputs DIR` end to end: DIR relative to the caller's cwd (the benchmark itself runs in a temporary
    directory), one timed step, and finite float arrays written after it."""
    import json
    import subprocess
    import numpy as np
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--batch", "1", "--seq", "256",
                        "--dump-outputs", "dump"], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-3000:]
    res = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])
    assert res["steps"] == 1
    got = {n: np.load(tmp_path / "dump" / f"{n}.npy") for n in ("loss", "params", "micro_batches", "count_grad_tot")}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in got.values())
    assert got["params"].shape == (1 << 22,) and got["loss"].shape == (1,)
    assert got["micro_batches"][0] >= res["config"]["micro_batches_timed"] and got["count_grad_tot"][0] >= 1


def test_launch_summary_parses_ncu_csv(tmp_path, capsys):
    ls = _load(os.path.join(ROOT, "tools", "launch_summary.py"), "launch_summary")
    csv = ('==PROF== noise\n"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC",'
           '"Section Name","Metric Name","Metric Unit","Metric Value"\n'
           '"0","1","python","h","void acco::ce_fwd_kernel(const __nv_bfloat16 *)","1","7","(512, 1, 1)","(8192, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","us","140.5"\n'
           '"1","1","python","h","void acco::ce_fwd_kernel(const __nv_bfloat16 *)","1","7","(512, 1, 1)","(8192, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","us","139.5"\n'
           '"2","1","python","h","nvjet_tst_192x256","1","7","(384, 1, 1)","(148, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","ns","20000"\n')
    p = tmp_path / "l.csv"
    p.write_text(csv)
    sys.argv = ["launch_summary.py", str(p)]
    ls.main()
    out = capsys.readouterr().out
    assert "3 launches, total 0.300 ms" in out and "x2" in out and "ce_fwd_kernel" in out


def test_memory_plan_tool():
    """tools/memory_plan.py: persistent buffers follow the arena / optimizer layout (6 bytes of bf16 buffers per parameter... x2 sets,
    16 bytes / W of fp32 shard); Llama-3-8B on 8 GPUs fits a 180 GB B200 with room to spare, on 1 GPU it does not."""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("memory_plan", os.path.join(root, "tools", "memory_plan.py"))
    mp = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mp)
    p8 = mp.main(["--model", "llama3-8b", "--gpus", "8", "--batch", "4", "--seq", "512"])
    assert p8["parameters"] == 8_030_261_248 and p8["fits_180gb"] and 60 < p8["total_gb"] < 120
    assert abs(p8["buffers_gb"]["optimizer shard: master, exp_avg, exp_avg_sq, stash (fp32)"] - 16 * p8["size_slice"] / 1e9) < 1e-9
    p1 = mp.main(["--model", "llama3-8b", "--gpus", "1", "--batch", "4", "--seq", "512"])
    assert not p1["fits_180gb"]
