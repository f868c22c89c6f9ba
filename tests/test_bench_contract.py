"""bench.py's reference arm (`--impl reference`) runs the CPU port of the reference algorithm and needs no
GPU: check that it prints ONE JSON line with the contract's keys (tiny configuration, ~1 s of CPU work).
`--dump-outputs`: the writer on CPU, the whole GPU arm on the device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_reference_arm(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-budget", "0.5", *extra], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    line = run_reference_arm("--n", "20", "--d", "20000")
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "aggregations/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["gpu_launches"] == 0 and line["vs_baseline"] is None
    # "reference" = the unmodified defences.py was found on this host (build container), "port" = oracle/ref_numpy.py
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "N=20" in line["metric"] and "N=20" in line["config"]["workload"]


def test_reference_arm_other_rules():
    for rule in ("TrimmedMean", "Bulyan", "NoDefense", "ALIE"):
        line = run_reference_arm("--rule", rule, "--n", "23", "--d", "4000", "--f", "5")
        assert rule in line["metric"] and line["value"] > 0


def test_reference_arm_port_when_no_checkout(tmp_path):
    """On the GPU box /root/reference does not exist: the arm must fall back to the NumPy port, same contract."""
    env = dict(os.environ, AFL_REFERENCE_DIR=str(tmp_path))
    code = ("import bench, json; bench.load_reference = lambda: (None, None); "
            "print(json.dumps(bench.cpu_reference_leg('Krum', 12, 3000, 2, budget=0.2)))")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    info = json.loads(out.stdout.strip().splitlines()[-1])
    assert info["kind"] == "port" and info["value"] > 0 and info["cores"] == 1


def test_cpu_legs_share_one_sample_shape():
    """VERDICT r1 weak #6: the two CPU figures of one record must be taken on the same D' and input distribution."""
    sys.path.insert(0, ROOT)
    import bench
    for rule, n, d in (("Krum", 100, 11_200_000), ("Bulyan", 500, 25_000_000), ("TrimmedMean", 1000, 10_000_000),
                       ("ALIE", 1000, 25_000_000)):
        a, b = bench.cpu_sample_dim(rule, n, d), bench.cpu_sample_dim(rule, n, d)
        assert a == b and 0 < a <= d
    g1, g2 = bench.cpu_inputs(7, 64, 5), bench.cpu_inputs(7, 64, 5)
    assert g1.dtype.name == "float32" and (g1 == g2).all()


def test_extra_configs_cover_the_baseline_configs():
    sys.path.insert(0, ROOT)
    import bench
    tags = [t[-1] for t in bench.extra_configs(1, 180.0)]
    assert tags == ["C3", "C4", "C5-krum", "C5-bulyan", "C5-alie"]
    full = {t[-1]: t for t in bench.extra_configs(1, 180.0)}
    assert full["C5-krum"][1:3] == (1000, 25_000_000)           # N=1000 x D=25M fp32 = 100 GB fits one B200
    small = {t[-1]: t for t in bench.extra_configs(1, 60.0)}
    assert small["C5-krum"][2] < 25_000_000                      # otherwise the largest D that fits, stated in the record


def test_clock_sampler_reads_only_samples_taken_after_align(tmp_path, monkeypatch):
    """bench.py's nvidia-smi sampler: `align()` returns right after a sample (so the following period is free of
    queries) and `stop()` reports only the samples taken from then on - checked with a stand-in `nvidia-smi` that
    prints one row per period: 1000 MHz before the timed region, 1965 MHz once a flag file exists."""
    import importlib.util
    import stat
    import time
    fake = tmp_path / "nvidia-smi"
    flag = tmp_path / "loaded"
    fake.write_text(f"""#!{sys.executable}
import os, sys, time
period = int(sys.argv[sys.argv.index("-lms") + 1]) / 1000.0
while True:
    mhz = 1965 if os.path.exists({str(flag)!r}) else 1000
    print(f"0, {{mhz}}, 1965, 700.0, Not Active, Not Active, Not Active, Active", flush=True)
    time.sleep(period)
""")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{tmp_path}{os.pathsep}{os.environ['PATH']}")
    monkeypatch.setenv("AFL_BENCH_CLOCKS_MS", "50")
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    s = bench.ClockSampler(0)
    assert s.period_ms == 50
    s.start()
    assert s.rows, "the first sample arrives before the timed region starts"
    s.align()
    flag.write_text("x")                     # "the step loop is running" from here on
    time.sleep(0.25)
    out = s.stop()
    assert out["samples"] >= 2 and out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"]
    # period 0 switches the sampler off (A/B runs): no process, and stop() says so
    monkeypatch.setenv("AFL_BENCH_CLOCKS_MS", "0")
    off = bench.ClockSampler(0)
    off.start(); off.align()
    assert off.stop()["sm_mhz"] is None


def test_dump_outputs_files_and_sample(tmp_path):
    """--dump-outputs: what the caller of each rule receives, float32 / float64 only; over the byte budget every vector is
    cut to the same seeded column sample, identical from run to run."""
    sys.path.insert(0, ROOT)
    import bench
    import numpy as np
    import torch
    from attacking_federate_learning_b200.sharded import ShardedAggregator

    class Cx:
        agg = ShardedAggregator()                   # one process: the vectors are already full length
    G = torch.arange(5 * 1000, dtype=torch.float32).reshape(5, 1000)
    cols, picks = bench.last_step_outputs(Cx, "Krum", G, 3, 1000)
    bench.write_outputs(str(tmp_path / "krum"), cols, picks)
    assert np.array_equal(np.load(tmp_path / "krum" / "aggregate.npy"), G[3].numpy())
    idx = np.load(tmp_path / "krum" / "krum_index.npy")
    assert idx.dtype == np.float64 and idx.tolist() == [3.0]
    cols, picks = bench.last_step_outputs(Cx, "Bulyan", G, (G[1] + 0.5, torch.tensor([4, 0, 2], dtype=torch.int32)), 1000)
    for run in ("b1", "b2"):
        bench.write_outputs(str(tmp_path / run), cols, picks, budget=2000)
        files = {p.name: np.load(p) for p in (tmp_path / run).iterdir()}
        assert set(files) == {"aggregate.npy", "bulyan_selection.npy", "columns.npy"}
        assert sum(p.stat().st_size for p in (tmp_path / run).iterdir()) <= 2000
        assert all(a.dtype in (np.float32, np.float64) for a in files.values())
        assert files["bulyan_selection.npy"].tolist() == [4.0, 0.0, 2.0]
        pos = files["columns.npy"].astype(np.int64)
        assert len(pos) > 50 and np.array_equal(files["aggregate.npy"], (G[1] + 0.5).numpy()[pos])
    for name in ("aggregate.npy", "columns.npy"):
        assert np.array_equal(np.load(tmp_path / "b1" / name), np.load(tmp_path / "b2" / name))


@pytest.mark.gpu
@pytest.mark.parametrize("rule", ["Krum", "Bulyan", "TrimmedMean", "ALIE"])
def test_dump_outputs_of_the_timed_path(tmp_path, rule):
    """Two runs with the same arguments write the same outputs; --steps is the number of timed steps."""
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import numpy as np
    n, d, f = 23, 40000, 5
    outs = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rule", rule, "--n", str(n), "--d", str(d),
                              "--f", str(f), "--steps", "4", "--warmup", "3", "--no-cpu-baseline", "--e2e-steps", "0",
                              "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600, cwd=ROOT,
                             env=dict(os.environ, AFL_BENCH_CLOCKS_MS="0"))
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
        assert line["steps"] == 4 and line["parity"]["match"]
        outs.append({p.name: np.load(p) for p in (tmp_path / run).iterdir()})
    a, b = outs
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    vec = a.pop("crafted.npy" if rule == "ALIE" else "aggregate.npy")
    assert vec.dtype == np.float32 and vec.shape == (d,) and np.isfinite(vec).all()
    want = {"Krum": {"krum_index.npy"}, "Bulyan": {"bulyan_selection.npy"}}.get(rule, set())
    assert set(a) == want and all(v.dtype == np.float64 for v in a.values())
    if rule == "Krum":
        assert 0 <= a["krum_index.npy"][0] < n
    if rule == "Bulyan":
        assert len(a["bulyan_selection.npy"]) == n - 2 * f
