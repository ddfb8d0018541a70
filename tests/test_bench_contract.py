"""bench.py contract checks that need no GPU: the reference arm (the C restatement of the step on the host cores) runs here and prints
the line the driver expects; both arms share one `config` object; the defaults are N = 1 with a K / W that finish in minutes."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("_bench_under_test", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "env_steps_per_sec" and line["unit"] == "env-steps/s"
    assert line["n_gpus"] == 1 and line["steps"] == 3 and line["warmup"] == 3 and line["higher_is_better"] is True
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["vs_baseline"] is None and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    bench = _bench_module()
    assert line["config"] == bench.config_of(16384, 1)                 # the GPU arm prints config_of(...) too: same_config
    assert "workload" in line["config"] and "model" not in line["config"]


def test_defaults_and_choices():
    bench = _bench_module()
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        a = bench.parse()
    finally:
        sys.argv = argv
    assert a.gpus == 1 and a.impl == "ours" and a.steps >= 20 and a.warmup >= 3 and a.envs == 16384
    assert a.metrics_collective == "peer" and a.dump_outputs is None
    assert bench.METRIC == "env_steps_per_sec" and bench.METRICS_EVERY == 16


def test_steps_and_dump_outputs_arguments_are_checked():
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and "error" in out.stderr, (argv, out.stderr[-2000:])


def test_dump_outputs_writes_float_arrays_and_a_fixed_sample_above_the_limit(tmp_path):
    """Files on disk, .npy headers included, stay within `max_bytes` (bench.py passes DUMP_MAX_BYTES // world to each rank)."""
    import numpy as np
    import torch
    bench = _bench_module()
    g = torch.Generator().manual_seed(0)
    n = 1000
    arrays = {"obs": torch.rand(n, 13, generator=g), "reset": torch.randint(0, 2, (n,), generator=g),
              "time_outs": torch.randint(0, 2, (n,), dtype=torch.uint8, generator=g)}
    whole = {"metrics": torch.rand(16, dtype=torch.float64, generator=g)}
    bench.dump_outputs(str(tmp_path / "all"), arrays, whole)
    got = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in (*arrays, *whole)}
    assert got["obs"].dtype == np.float32 and got["reset"].dtype == got["time_outs"].dtype == got["metrics"].dtype == np.float64
    for k, t in {**arrays, **whole}.items():
        assert np.array_equal(got[k], t.numpy()), k
    headers = sum(os.path.getsize(tmp_path / "all" / f"{k}.npy") - got[k].nbytes for k in got)
    cap = headers + whole["metrics"].numpy().nbytes + 100 * (13 * 4 + 8 + 8)      # room for 100 of the 1000 rows
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), arrays, whole, "_rank1", max_bytes=cap)
    s1 = {k: np.load(tmp_path / "s1" / f"{k}_rank1.npy") for k in got}
    s2 = {k: np.load(tmp_path / "s2" / f"{k}_rank1.npy") for k in got}
    assert sum(os.path.getsize(tmp_path / "s1" / f) for f in os.listdir(tmp_path / "s1")) <= cap and len(s1["obs"]) == 100
    assert np.array_equal(s1["metrics"], got["metrics"])
    rows = np.flatnonzero((arrays["obs"].numpy()[:, None, :] == s1["obs"][None]).all(-1).any(-1))     # the rows that were kept
    assert len(rows) == 100
    for k, t in arrays.items():
        assert np.array_equal(s1[k], s2[k]) and np.array_equal(s1[k], t.numpy()[rows].astype(s1[k].dtype)), k
