"""The bench.py JSON contract, checked on the committed lines of the last GPU runs (profiles/r02_*.json): every key the driver and
the judge read is present with the right type, the derived numbers are self-consistent, and the reference arm mirrors the b200 arm's
metric / unit / config."""
import json
import os

import pytest

PROFILES = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles")


def _load(name):
    path = os.path.join(PROFILES, name)
    if not os.path.exists(path):
        pytest.skip("%s not committed" % name)
    return [json.loads(l) for l in open(path) if l.startswith("{")]


def _check_common(d):
    for k, t in (("metric", str), ("value", float), ("unit", str), ("n_gpus", int), ("steps", int), ("warmup", int), ("ms_per_step", float),
                 ("higher_is_better", bool), ("scaling", str), ("dtype", str), ("data", str), ("config", dict), ("e2e", dict)):
        assert k in d and isinstance(d[k], t), (k, type(d.get(k)))
    assert "vs_baseline" in d and d["vs_baseline"] is None          # BASELINE.md holds no published number for this metric
    assert d["warmup"] >= 3 and d["scaling"] == "weak" and d["data"] == "synthetic" and d["higher_is_better"] is True
    assert "workload" in d["config"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k


@pytest.mark.parametrize("name", ["r02_bench.json", "r02_scale_n2.json"])
def test_b200_arm_line(name):
    d = _load(name)[-1]
    _check_common(d)
    assert d["gpu_launches"] > 0
    assert abs(d["value"] - d["n_gpus"] * d["steps"] / (d["ms_per_step"] * d["steps"] * 1e-3)) / d["value"] < 1e-6
    assert d["e2e"]["h2d_bytes_per_step"] >= 480 * 640 * 3 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["e2e"]["value"] != d["value"]                          # measured separately, not a copy of the device-timed number
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    assert [x["kernel"] for x in d["rooflines"]][0] == r["kernel"] and len(d["rooflines"]) >= 3
    c = d["clocks"]
    assert c["sm_mhz"] > 0.9 * c["sm_max_mhz"] and not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if d["n_gpus"] == 1:
        b = d["cpu_baseline"]
        for k in ("value", "unit", "cores", "kind", "sample"):
            assert k in b, k
        assert b["kind"] in ("reference", "port") and b["unit"] == d["unit"] and b["value"] < d["value"]


@pytest.mark.parametrize("name,arm", [("r02_bench_reference_arm.json", "r02_bench.json"), ("r02_scale_n2_reference.json", "r02_scale_n2.json")])
def test_reference_arm_line_mirrors_the_b200_arm(name, arm):
    r, d = _load(name)[-1], _load(arm)[-1]
    _check_common(r)
    assert r["impl"] == "reference" and r["gpu_launches"] == 0
    for k in ("metric", "unit", "higher_is_better", "config", "n_gpus"):
        assert r[k] == d[k], k
    assert r["e2e"]["value"] == r["value"] and r["e2e"]["h2d_bytes_per_step"] == 0 and r["e2e"]["d2h_bytes_per_step"] == 0
    b = r["cpu_baseline"]
    assert b["value"] == r["value"] and b["kind"] in ("reference", "port") and b["cores"] >= r["n_gpus"]


def test_other_configuration_lines():
    lines = _load("r02_bench_other_configs.jsonl")
    assert len(lines) == 3
    for d in lines:
        _check_common(d)
        assert d["value"] > d["torch_cuda_baseline"]["value"] > 0 and d["cpu_baseline"]["value"] > 0


def test_eco_rows_of_the_roofline_list():
    """bench.py appends the ECO rows (tools/eco_bench.py in a subprocess) to `rooflines[]`: without a GPU the row says so instead of
    raising; with the tool's output (on a machine with a GPU, or the recorded data below) it carries the roofline keys."""
    import torch
    import bench
    peaks = {"hbm_gbs": 6572.2}
    rows = bench.eco_rows(peaks)
    if torch.cuda.is_available():
        assert rows and all("unavailable" not in r and r["bound"] == "hbm" and r["peak"] == peaks["hbm_gbs"] for r in rows), rows
    else:
        assert len(rows) == 1 and "unavailable" in rows[0]                   # no CUDA device here
    data = {"deep 15x8 x 200 x 64": {"us_median": 40.0, "us_min": 39.0, "sample_memory_bytes": 12288000, "reference_sweep_bytes": 147456000,
                                     "GBps_vs_one_read": 307.2, "GBps_vs_reference_sweeps": 3686.4},
            "joint deep 15x8 x 30 x 256 -> 64": {"us_median": 2000.0, "us_min": 1990.0, "gn_x_cg": "10 x 10", "sample_bytes": 7372800},
            "scores 5 scales": {"us_median": 30.0, "us_min": 29.0, "bytes": 3000000, "launches": 4}}
    rows = bench.eco_rows_from(data, peaks)
    assert len(rows) == 3
    for r in rows:
        assert {"kernel", "bound", "achieved", "peak", "unit", "frac", "traffic", "us_per_launch", "algorithmic_bytes"} <= set(r)
        assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(rows[0]["achieved"] - 12288000 / 40e-6 / 1e9) < 1e-6
