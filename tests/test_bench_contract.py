"""The parts of the bench.py contract that run without a GPU: the reference arm (the oracle port timed on the
host cores) prints ONE JSON line with the keys the driver reads, and the roofline accounting counts the flop the
SYRK executes (n minus the folded slack columns), not the structure-blind figure."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_for_the_smallest_config():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ipm_iterations_per_s" and d["unit"] == "iterations/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and abs(d["ms_per_iteration"] - 1000.0 / d["value"]) < 1e-6 and d["ms_per_step"] > 0
    assert d["details"]["iterations_timed"] >= 1          # REAL iterations of the oracle's loop, not a cost model
    assert "real iterations" in d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.bench_config("C1", 512, 1024, 0, 1)    # the product arm prints the same dict
    assert d["e2e"] == {"value": d["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "C1" in d["config"]["workload"] and d["dtype"] == "f64" and d["vs_baseline"] is None


def test_reference_arm_is_silent_on_non_zero_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--workload", "C1", "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_roofline_counts_executed_flop():
    sys.path.insert(0, ROOT)
    import bench
    m, n = 16384, 32768
    prof = {"syrk_ms": 2 * 24 * 190.0, "syrk_launches": 48, "potrf_ms": 2 * 24 * 55.0, "potrf_launches": 48,
            "syrk_cols": 2 * 24576, "solves": 2}
    r = bench._roofline(prof, m, n)
    assert r["syrk_cols"] == 24576 and r["bound"] == "tensor" and r["unit"] == "TFLOP/s"
    assert abs(r["flop_per_launch"] - m * (m + 1) * 24576.0) < 1.0
    assert abs(r["achieved"] - m * (m + 1) * 24576.0 / 0.190 * 1e-12) < 1e-9
    assert abs(r["frac"] - r["achieved"] / 40.0) < 1e-12
    assert r["algorithmic_tflops"] > r["achieved"]                       # structure-blind count, reported beside it
    assert r["traffic"] == bench.SYRK_TRAFFIC[(m, 24576)][0]             # ncu capture of this exact shape ...
    assert r["traffic_source"].startswith("profiles/")                   # ... labelled as such, not measured in the run
    assert bench._roofline(prof, 4096, 8192)["traffic"] is None          # no capture -> null, not a guess
    rm = bench._roofline(prof, m, n, peak_measured=36.9)
    assert rm["peak"] == 40.0 and rm["peak_measured"] == 36.9 and abs(rm["frac_of_measured"] - rm["achieved"] / 36.9) < 1e-12


def test_both_arms_share_one_config_dict():
    sys.path.insert(0, ROOT)
    import bench
    for wl, (m, n) in bench.WORKLOADS.items():
        for world in (1, 8):
            c = bench.bench_config(wl, m, n, 0, world)
            assert set(c) == {"workload", "parallelism", "l2"} and wl in c["workload"]


def _bench(*argv, timeout=120):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(argv), capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_steps_warmup_and_dump_outputs_are_validated(tmp_path):
    for argv in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r = _bench(*argv)
        assert r.returncode == 2 and "error:" in r.stderr, (argv, r.stderr[-2000:])
    assert not (tmp_path / "d").exists()


def test_dump_outputs_writes_float64_npy_within_the_limit(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    bench.dump_outputs(str(tmp_path / "d"), {"x": np.arange(5, dtype=np.float32), "fun": -1.5, "iteration": 14})
    got = {f: np.load(str(tmp_path / "d" / f)) for f in sorted(os.listdir(tmp_path / "d"))}
    assert sorted(got) == ["fun.npy", "iteration.npy", "x.npy"]
    assert all(a.dtype == np.float64 for a in got.values())
    np.testing.assert_array_equal(got["x.npy"], np.arange(5.0))
    assert got["fun.npy"] == -1.5 and got["iteration.npy"] == 14.0
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 8 + 1)})
    assert not (tmp_path / "big").exists()


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_solve(tmp_path):
    """The product arm on C1 (two timed solves): x, fun and iteration as a caller of `solve_resident` receives them,
    within the parity bar of the committed oracle fixture."""
    out = tmp_path / "out"
    r = _bench("--workload", "C1", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-e2e",
               "--dump-outputs", str(out), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 2 and d["warmup"] == 1
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "oracle_C1_seed0.json")))
    x = np.load(str(out / "x.npy"))
    fun, it = float(np.load(str(out / "fun.npy"))), float(np.load(str(out / "iteration.npy")))
    assert x.dtype == np.float64 and x.shape == (768,)
    assert np.abs(x - np.load(os.path.join(ROOT, "tests", "golden", gold["x_file"]))).max() <= 1e-6
    assert abs(it - gold["iterations"]) <= 1 and it == d["details"]["iterations_per_solve"]
    assert abs(fun - gold["fun"]) <= 1e-8 * abs(gold["fun"]) and fun == d["details"]["objective"]
