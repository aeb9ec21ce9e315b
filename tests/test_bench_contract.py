"""bench.py's output contract: exactly ONE JSON line on stdout with the keys the driver reads.  The reference arm
(the unmodified reference on the host's cores) runs without a GPU; our arm is a `-m gpu` test on the small
BASELINE configs[0]-shaped workload."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers

BENCH = os.path.join(helpers.ROOT, "bench.py")
COMMON = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
          "data", "config", "e2e", "cpu_baseline"}


def _run(args, tmp_path):
    p = subprocess.run([sys.executable, BENCH, "--data-dir", os.path.join(helpers.DATA_ROOT, "bench")] + args,
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, f"stdout must carry one line, got {len(lines)}: {p.stdout[:500]}"
    return json.loads(lines[0])


def test_reference_arm_line(tmp_path):
    if not os.path.exists(helpers.ref_bin("ema")):
        pytest.skip("oracle/_ref/ema missing")
    d = _run(["--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0"], tmp_path)
    assert d["impl"] == "reference" and COMMON <= set(d)
    assert d["value"] > 0 and d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.gpu
def test_our_arm_line(tmp_path):
    dump = tmp_path / "outputs"
    d = _run(["--workload", "c1", "--steps", "2", "--warmup", "3", "--dump-outputs", str(dump)], tmp_path)
    assert "impl" not in d or d["impl"] != "reference"
    assert COMMON | {"roofline", "clocks", "gpu_launches"} <= set(d)
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0 and d["scaling"] == "weak" and d["n_gpus"] == 1 and d["steps"] == 2
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    c = d["cpu_baseline"]
    if os.path.exists(helpers.ref_bin("ema")):
        assert c["kind"] == "reference" and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    else:   # without a built reference the line says so instead of carrying a number
        assert c["kind"] == "reference" and c["value"] is None and c["unavailable"]
    # --dump-outputs: one float64 column per SAM field, one row per record of the last timed bucket (one per read)
    cols = {f: np.load(dump / f"sam_{f}.npy") for f in ("flag", "rname", "pos", "mapq", "tlen", "XG", "line_crc32")}
    assert all(v.dtype == np.float64 and v.shape == (2 * d["config"]["bucket_pairs"],) for v in cols.values())
    assert (cols["pos"] > 0).mean() > 0.9 and np.isfinite(cols["XG"]).any() and len(np.unique(cols["line_crc32"])) > 0.99 * len(cols["pos"])
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    m = d["sw_microbench"]
    assert "error" not in m, m
    assert m["qlen"] == 151 and m["gcups_visited"] > 100 and 0.05 < m["roofline"]["frac"] < 1 and m["roofline"]["bound"] == "int-alu"
