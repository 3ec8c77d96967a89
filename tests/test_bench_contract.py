"""bench.py's output contract: the committed round line (profiles/r1/bench_r1_bf16.json, produced on a B200 by the default
`python bench.py`) and the live `--impl reference` line carry every key the driver reads, with consistent values."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"]


def _check_common(line):
    for k in BASE_KEYS:
        assert k in line, k
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "reasoning" in line["metric"] and "reasoning steps/sec" in base["metric"]
    assert line["higher_is_better"] is True and line["scaling"] == "weak" and line["data"] == "synthetic"
    assert line["vs_baseline"] is None                       # BASELINE.json publishes no number for this metric
    assert "workload" in line["config"] and "model" not in line["config"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in line["e2e"], k
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in line["cpu_baseline"], k
    assert line["cpu_baseline"]["kind"] in ("reference", "port")


def test_committed_gpu_line_has_the_full_contract():
    line = json.load(open(os.path.join(ROOT, "profiles", "r1", "bench_r1_bf16.json")))
    _check_common(line)
    assert line["n_gpus"] == 1 and line["dtype"] == "bf16" and line["warmup"] >= 3
    L = 12
    assert abs(line["value"] - line["steps"] * L / (line["ms_per_step"] * 1e-3 * line["steps"])) < 1e-6 * line["value"]
    assert line["gpu_launches"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["e2e"]["value"] < line["value"]              # the copies are inside the timed region
    for k in ("sm_mhz", "sm_max_mhz", "reasons"):
        assert k in line["clocks"], k
    assert not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    for roof in (line["roofline"], line["roofline_kb_attend"]):
        for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
            assert k in roof, k
        assert roof["bound"] in ("hbm", "tensor") and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
        assert roof["traffic"] is not None                   # ncu dram bytes of the committed captures (profiles/traffic.json)
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else None
    if peaks:
        assert line["roofline_kb_attend"]["peak"] == peaks["hbm_gbs"]


def test_reference_arm_line_live():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    _check_common(line)
    assert line["impl"] == "reference" and line["dtype"] == "f32"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["e2e"]["value"] == line["value"] == line["cpu_baseline"]["value"]
    assert line["cpu_baseline"]["cores"] >= 1


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(tmp_path):
    """`--steps K` times exactly K passes (one block), and `--dump-outputs` writes what the last of them returned: two runs
    with the same arguments write the same arrays."""
    from mac_network_b200.synthetic import SHAPES
    B, S, N, d, L = SHAPES["headline"]
    shapes = {"control": (B, d), "memory": (B, d), "att_kb": (L, B, N), "att_question": (L, B, S)}
    dumps = []
    for run in range(2):
        out_dir = str(tmp_path / ("run%d" % run))
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--skip-train",
                              "--skip-cpu", "--dump-outputs", out_dir], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-800:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == 3 and line["timed_blocks"]["resident"]["blocks"] == 1
        assert sorted(os.listdir(out_dir)) == sorted(k + ".npy" for k in shapes)
        dumps.append({k: np.load(os.path.join(out_dir, k + ".npy")) for k in shapes})
    for k, shape in shapes.items():
        assert dumps[0][k].dtype == np.float32 and dumps[0][k].shape == shape, k
        assert np.isfinite(dumps[0][k]).all(), k
        assert np.array_equal(dumps[0][k], dumps[1][k]), k
    for k in ("att_kb", "att_question"):
        assert np.allclose(dumps[0][k].sum(-1), 1.0, atol=1e-5), k
