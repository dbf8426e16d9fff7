"""The driver's bench.py contract: one JSON line with the agreed keys, for both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "bench.py must print exactly ONE line on stdout"
    return json.loads(lines[0])


def test_reference_arm_json_contract(tmp_path):
    """--impl reference runs without a GPU: the reference's CPU path on the host cores, bounded sample."""
    d = _run(["--impl", "reference", "--grid", "32", "--ref-planes", "4", "--steps", "2", "--warmup", "1",
              "--dump-outputs", str(tmp_path)])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["value"] > 0 and d["unit"] == "points/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None
    # --dump-outputs: the last timed step ran on 32 x 32 x 4 planes; the same seeded inputs give the same losses again
    assert sorted(os.listdir(tmp_path)) == ["loss.npy"]
    loss = np.load(tmp_path / "loss.npy")
    assert loss.dtype == np.float32 and loss.shape == (2,) and np.all(loss > 0)
    again = tmp_path / "again"
    _run(["--impl", "reference", "--grid", "32", "--ref-planes", "4", "--steps", "2", "--warmup", "1",
          "--dump-outputs", str(again)])
    assert np.array_equal(np.load(again / "loss.npy"), loss)


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=60, cwd=ROOT)
    assert r.returncode != 0 and "--steps" in r.stderr and not r.stdout.strip()


@pytest.mark.gpu
def test_b200_arm_json_contract(tmp_path):
    d = _run(["--grid", "64", "--steps", "4", "--warmup", "3", "--no-extra", "--dump-outputs", str(tmp_path)])
    assert BASE_KEYS | {"clocks", "roofline"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] >= 3 and d["gpu_launches"] == 4
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and "workload" in d["config"] and "l2" in d["config"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in d["roofline"]
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"]
    assert d["e2e"]["h2d_bytes_per_step"] == 4 * (64 * 4 + 64 + 4 * 64 + 4) and d["e2e"]["d2h_bytes_per_step"] == 16
    assert 0 < d["e2e"]["value"] <= d["value"] * 1.05
    for k in ("sm_mhz", "sm_max_mhz", "reasons"):
        assert k in d["clocks"]
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in d["cpu_baseline"]
    # the two loss values of the timed path and of the end-to-end path agree
    assert d["e2e"]["loss"] == [d["loss"]["sigma"], d["loss"]["u"]]
    # --dump-outputs: the last timed step's sums and losses, the losses being the ones the JSON line reports
    assert sorted(os.listdir(tmp_path)) == ["loss.npy", "sums.npy"]
    sums, loss = np.load(tmp_path / "sums.npy"), np.load(tmp_path / "loss.npy")
    assert sums.dtype == np.float64 and sums.shape == (2,) and np.all(sums > 0)
    assert loss.dtype == np.float32 and loss.tolist() == [d["loss"]["sigma"], d["loss"]["u"]]
    assert loss.tolist() == [float(np.float32(s * (1.0 / 64 ** 3))) for s in sums]   # weights (1, 1): L = float(acc * (1/N))
