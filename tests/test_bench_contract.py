"""The committed bench line of the round (profiles/) keeps the driver's JSON contract: a change to bench.py that drops a
key shows here without a GPU."""
import glob
import json
import os

import pytest

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
LINES = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_bench_n*_512_*.json")))


@pytest.mark.parametrize("path", LINES, ids=[os.path.basename(p) for p in LINES])
def test_bench_line_contract(path):
    d = json.loads(open(path).read().strip().splitlines()[-1])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    # BASELINE.json: "voxels/s full-texture voxel-based on 512^3 @1/2/4/8 B200; %HBM roofline" -- the line carries the
    # quantity, the "@N B200" part is n_gpus and the roofline part is the `roofline` object
    assert base["metric"].startswith(d["metric"])
    assert d["unit"] == "voxels/s" and d["higher_is_better"] is True and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] >= 1 and d["warmup"] >= 3
    assert d["scaling"] in ("weak", "strong") and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["gpu_launches"] > 0
    c = d["clocks"]
    assert c["sm_mhz"] and c["sm_max_mhz"] and not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s")
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"])
    if d["n_gpus"] == 1 and d.get("cpu_baseline"):
        b = d["cpu_baseline"]
        assert b["kind"] in ("reference", "port") and b["cores"] >= 1 and b["value"] > 0 and b["sample"]


def test_at_least_one_line_is_committed():
    assert LINES


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(tmp_path):
    """--dump-outputs writes one float64 [features, voxels] array per class, 64 MB at most, and two runs with the same
    arguments write the same values; --steps is the number of timed steps the line reports"""
    import subprocess
    import sys

    import numpy as np
    n_features = {"glcm": 24, "glrlm": 16, "glszm": 16, "gldm": 14, "ngtdm": 5}
    dumps = []
    for run, steps in enumerate((1, 2)):
        out = tmp_path / f"run{run}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                            "--size", "40", "--no-e2e", "--no-secondary", "--no-cpu-baseline", "--no-numa-bind",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == steps
        files = sorted(os.listdir(out))
        assert files == sorted(f"{c}.npy" for c in n_features)
        assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
        d = {f[:-4]: np.load(out / f) for f in files}
        for c, a in d.items():
            assert a.dtype == np.float64 and a.shape == (n_features[c], 40 ** 3)
        dumps.append(d)
    for c in n_features:
        assert np.array_equal(dumps[0][c], dumps[1][c], equal_nan=True), c
