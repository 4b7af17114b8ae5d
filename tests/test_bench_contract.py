"""The bench line contract (driver-facing): checked on the most recent committed GPU bench lines under profiles/ and, for the
reference arm, by running it here on a tiny sample (it is CPU-only)."""
import glob
import json
import os
import subprocess
import sys

import pytest

from oracle import ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e"}


def _latest(pattern):
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    assert files, pattern
    return json.load(open(files[-1]))


def _check_common(j):
    assert BASE_KEYS <= set(j), BASE_KEYS - set(j)
    assert j["metric"] == "pdas_path_cv_fits_per_sec" and j["unit"] == "fits/s" and j["higher_is_better"] is True
    assert j["dtype"] == "f64" and j["data"].startswith("synthetic") and j["vs_baseline"] is None  # BASELINE.md publishes no number
    assert "workload" in j["config"] and "model" not in j["config"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(j["e2e"])
    assert j["scaling"] in ("weak", "strong")


def test_our_bench_line_single_gpu():
    j = _latest("r0*_bench.json")
    _check_common(j)
    assert j["n_gpus"] == 1 and j["warmup"] >= 3 and j["gpu_launches"] > 0
    assert abs(j["value"] - 220 * 1e3 / j["ms_per_step"]) < 1e-6 * j["value"]  # 220 fits per step
    assert j["e2e"]["h2d_bytes_per_step"] >= 8 * 1000 * 500000 and j["e2e"]["value"] < j["value"]
    r = j["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] >= r["algorithmic_bytes_per_launch"]  # DRAM traffic from ncu is never below the algorithmic bytes
    c = j["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] == "reference" and c["cores"] >= 1
    k = j["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(k)
    assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(k["reasons"]))


def test_our_bench_lines_multi_gpu_are_weak_scaling_on_unique_fits():
    for n in (2, 4, 8):
        j = _latest(f"r0*_bench_n{n}.json")
        _check_common(j)
        assert j["n_gpus"] == n and j["scaling"] == "weak"
        assert j["fits_per_step"] == 20 * (1 + 10 * n)  # the full-data chain is counted once, not once per rank
        assert abs(j["value"] - j["fits_per_step"] * 1e3 / j["ms_per_step"]) < 1e-6 * j["value"]
        assert j["e2e"]["h2d_bytes_per_step"] < 8 * 1000 * 500000  # every rank uploads only its column shard


@pytest.mark.skipif(not ref.available(), reason="the reference's own library (oracle/_ref, built by oracle/Makefile from the "
                                               "original project's sources, which are not part of this repository) is not built")
def test_reference_arm_runs_here_and_keeps_the_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env=dict(os.environ, BESS_BENCH_REF_LEVELS="1", BESS_BENCH_REF_PROCS="2"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1  # exactly one JSON line on stdout
    j = json.loads(lines[0])
    _check_common(j)
    assert j["impl"] == "reference" and j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    assert j["cpu_baseline"]["kind"] == "reference" and j["cpu_baseline"]["cores"] >= 1 and j["e2e"]["value"] == j["value"]


def test_committed_reference_arm_line_ran_config_5_itself():
    """The reference arm of the last GPU-box run (profiles/r0*_bench_ref.json): from round 2 on it times the reference on
    config 5 itself (n=1000, p=500000, 220 fits per call), one call per process, not a proportional slice."""
    j = _latest("r0*_bench_ref.json")
    _check_common(j)
    assert j["impl"] == "reference" and j["config"]["same_config_as_gpu_arm"] is True
    assert "p=500000" in j["config"]["reference_sample"] and "s.list=1..20" in j["config"]["reference_sample"]
    assert j["steps"] >= 1 and j["cpu_baseline"]["cores"] >= 1
    assert abs(j["value"] - 220 * j["cpu_baseline"]["cores"] / j["cpu_baseline"]["seconds"]) < 1e-6 * j["value"]
