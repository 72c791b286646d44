"""bench.py against the driver's contract: ONE JSON line on stdout with the required keys, the reference arm on the host cores
(rank 0 only under torchrun), a loud failure of the native arm without a GPU, and -- on the B200 box -- the native line with
`roofline`, `clocks`, `e2e` and a non-zero `gpu_launches`."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "cpu_baseline", "gpu_launches"}


def run_bench(*args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, timeout=timeout, env=e, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-units", "8")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "audio-sec/sec (MFCC+spectral feats)" and d["unit"] == "audio-s/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f64"
    assert d["config"]["workload"].startswith("cfg4")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "8 x 2.0 s segments" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    r = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_native_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    r = run_bench("--steps", "1", "--warmup", "3", "--no-cpu")
    assert r.returncode != 0 and r.stdout.strip() == ""
    assert "no CUDA device" in r.stderr and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_native_line_on_the_gpu():
    r = run_bench("--hours", "0.1", "--steps", "2", "--warmup", "3", "--no-cpu", "--e2e-steps", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert (BASE_KEYS - {"cpu_baseline"}) <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["dtype"] == "f32" and d["scaling"] == "strong"
    assert d["gpu_launches"] > 0 and d["value"] > 1e5
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and rf["peak"] > 1000 and 0 < rf["frac"] < 1
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    e = d["e2e"]
    n_seg = d["config"]["segments"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == int(0.1 * 3600 * 44100) * 2 and e["d2h_bytes_per_step"] == n_seg * 24 * 8
    assert e["matches_device_path"] is True and e["f32"]["h2d_bytes_per_step"] == int(0.1 * 3600 * 44100) * 4
    assert d["weak"]["value"] > 1e5 and d["roofline"]["aggregate_ms_per_step"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("wl,extra", [("cfg3", ["--units", "4000"]), ("cfg2", ["--units", "512", "--nfft", "512,2048"]), ("cfg5", ["--seconds", "20"])])
def test_secondary_workloads_on_the_gpu(wl, extra):
    """cfg2 / cfg3 / cfg5 under the same one-line contract (roofline + clocks + e2e)."""
    r = run_bench("--workload", wl, "--steps", "2", "--warmup", "3", "--no-cpu", "--e2e-steps", "1", *extra)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert (BASE_KEYS - {"cpu_baseline"}) <= set(d) and d["config"]["workload"].startswith(wl)
    assert d["value"] > 0 and d["gpu_launches"] > 0 and 0 < d["roofline"]["frac"] < 1.2 and d["e2e"]["value"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    if wl == "cfg2":
        assert [s["n_fft"] for s in d["roofline"]["sweep"]] == [512, 2048]


def test_bad_step_counts_and_reference_dump_are_refused():
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = run_bench(*args)
        assert r.returncode == 2 and r.stdout.strip() == "" and "error:" in r.stderr, args


def test_dump_outputs_keeps_a_seeded_sample_under_the_budget(tmp_path):
    import importlib.util
    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench_module", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    a = torch.arange(1000 * 6, dtype=torch.float64).reshape(1000, 6)
    b = torch.arange(1000 * 10, dtype=torch.float32).reshape(1000, 10)
    bench.dump_outputs(str(tmp_path / "all"), {"a": a, "b": b})
    assert np.array_equal(np.load(tmp_path / "all" / "a.npy"), a.numpy()) and np.load(tmp_path / "all" / "b.npy").dtype == np.float32
    budget = (a.numel() * 8 + b.numel() * 4) // 4
    for run in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / run), {"a": a, "b": b}, budget=budget)
    sa, sb = np.load(tmp_path / "s1" / "a.npy"), np.load(tmp_path / "s1" / "b.npy")
    assert sa.nbytes + sb.nbytes <= budget and sa.shape == (250, 6) and sb.shape == (250, 10)
    rows = sa[:, 0] / 6
    assert np.all(np.diff(rows) > 0) and np.array_equal(sb[:, 0] / 10, rows)       # same units in both, ascending
    assert np.array_equal(np.load(tmp_path / "s2" / "a.npy"), sa)
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path / "i"), {"i": torch.zeros(3, dtype=torch.int32)})


@pytest.mark.gpu
def test_dump_outputs_of_two_runs_agree(tmp_path):
    """--dump-outputs writes the [segments, 24] float64 vectors of the last timed step; the same arguments give the same inputs, so
    runs of one build write the same values, whatever the number of steps.  --steps sets the steps actually timed: twice the steps,
    twice the kernel launches in the timed window."""
    import numpy as np
    outs, launches = [], []
    for run, steps in (("a", 3), ("b", 6)):
        r = run_bench("--hours", "0.05", "--steps", str(steps), "--warmup", "1", "--no-cpu", "--no-e2e", "--no-weak",
                      "--dump-outputs", str(tmp_path / run))
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip().splitlines()[-1])
        assert d["steps"] == steps
        launches.append(d["gpu_launches"])
        assert sorted(os.listdir(tmp_path / run)) == ["features.npy"]
        outs.append(np.load(tmp_path / run / "features.npy"))
        assert outs[-1].dtype == np.float64 and outs[-1].shape == (d["config"]["segments"], 24)
        assert abs(float(np.nansum(outs[-1])) - d["checksum"]) <= 1e-9 * abs(d["checksum"])
    np.testing.assert_array_equal(outs[0], outs[1])
    assert launches[0] > 0 and launches[1] == 2 * launches[0], launches


@pytest.mark.gpu
def test_dump_outputs_sample_a_large_output_on_the_device(tmp_path):
    """cfg3 with 16 000 clips computes [16000, 13, 101] float32 (84 MB): the dump keeps the same seeded sample of clips in every run,
    under 64 MB."""
    import numpy as np
    outs = []
    for run in ("a", "b"):
        r = run_bench("--workload", "cfg3", "--units", "16000", "--steps", "2", "--warmup", "1", "--no-cpu", "--no-e2e",
                      "--dump-outputs", str(tmp_path / run))
        assert r.returncode == 0, r.stderr[-2000:]
        f = tmp_path / run / "features.npy"
        assert sorted(os.listdir(tmp_path / run)) == ["features.npy"] and os.path.getsize(f) < 64_000_000
        outs.append(np.load(f))
        assert outs[-1].dtype == np.float32 and 10000 < outs[-1].shape[0] < 16000 and outs[-1].shape[1:] == (13, 101)
        assert np.isfinite(outs[-1]).all()
    np.testing.assert_array_equal(outs[0], outs[1])


@pytest.mark.parametrize("wl", ["cfg3", "cfg2", "cfg5"])
def test_reference_arm_secondary_workloads(wl):
    r = run_bench("--impl", "reference", "--workload", wl, "--steps", "1", "--warmup", "0", "--cpu-units", "8")
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["value"] > 0 and d["config"]["workload"].startswith(wl) and d["cpu_baseline"]["kind"] == "port"
