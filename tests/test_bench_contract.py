"""bench.py contract (CPU part): the reference arm prints ONE JSON line with the keys the driver
reads, and the cost-model extrapolation is self-consistent.  (The GPU arm is exercised under
gpurun; its JSON lines are committed under profiles/.)"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json(monkeypatch, capsys):
    import bench
    real = bench.run_cpu_sample
    monkeypatch.setattr(bench, "run_cpu_sample", lambda n_s=None, reps=1: real(512, reps))
    args = type("A", (), dict(gpus=1, steps=2, warmup=1))()
    bench.reference_main(args)
    line = capsys.readouterr().out.strip().splitlines()[-1]
    d = json.loads(line)
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"]


def test_non_zero_ranks_of_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="3", WORLD_SIZE="8", LOCAL_RANK="3")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "8"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_extrapolation_model():
    import bench
    t = dict(assemble=1.0, chol=2.0, solve=0.5, posterior=3.0)
    # doubling N: assemble x4, chol x8, solves x4, posterior x4 (x N*/N* ratio)
    assert np.isclose(bench.cpu_extrapolate(t, 100, 10, 200, 10), 4 + 16 + 2 + 12)
    assert np.isclose(bench.cpu_extrapolate(t, 100, 10, 100, 20), 1 + 2 + 0.5 + 6)


def test_dump_outputs_float64_and_bounded_sample(tmp_path, monkeypatch):
    import bench
    mean, var = np.arange(1000, dtype=np.float64), np.arange(1000, dtype=np.float32) * 0.5
    bench.dump_outputs(str(tmp_path / "full"), logpdf=np.float64(-3.5), mean=mean, var=var)
    got = {p.stem: np.load(p) for p in (tmp_path / "full").iterdir()}
    assert sorted(got) == ["logpdf", "mean", "var"] and all(a.dtype == np.float64 for a in got.values())
    assert got["logpdf"] == -3.5 and np.array_equal(got["mean"], mean) and np.array_equal(got["var"], var)
    # above the limit: the same seeded sample of entries every time, within the limit, indices included
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), logpdf=np.float64(-3.5), mean=mean, var=var)
    a, b = ({p.stem: np.load(p) for p in (tmp_path / d).iterdir()} for d in ("a", "b"))
    assert sorted(a) == ["logpdf", "mean", "sample_index", "var"]
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.nbytes for v in a.values()) <= 4000
    idx = a["sample_index"].astype(np.int64)
    assert np.array_equal(a["mean"], mean[idx]) and np.array_equal(a["var"], var[idx])


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_committed_gpu_bench_line_has_contract_keys():
    d = json.loads(open(os.path.join(ROOT, "profiles", "bench_r1_1gpu.json")).read().strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert k in d, k
    assert d["roofline"]["bound"] == "tensor" and 0 < d["roofline"]["frac"] <= 1.05
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["gpu_launches"] > 0 and d["warmup"] >= 3
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
