"""bench.py's reference arm runs without a GPU (it is what the driver launches with `--impl reference`): the JSON
contract of its line, for the default workload and for the reference's own CPU case (configs[0])."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", *extra],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout                      # ONE JSON line on stdout
    return json.loads(lines[0])


@pytest.mark.parametrize("extra,config", [((), 2), (("--config", "0"), 0)])
def test_reference_arm_line(extra, config):
    d = _run(*extra)
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("IK-solved frames/sec") and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert f"configs[{config}]" in d["config"]["workload"]
    if config == 0:
        assert d["latency_us"]["per_window_mean"] > 0


def test_reference_arm_dumps_its_last_step(tmp_path, golden):
    """--dump-outputs: float32 .npy files of the last timed step, identical from run to run (configs[0]: the dance
    windows, whose poses the reference's own modules produced in tests/golden/dance.npz)."""
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        _run("--config", "0", "--dump-outputs", str(tmp_path / run))
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("poses", "joints")})
    a, b = dumps
    assert a["poses"].dtype == np.float32 and a["poses"].shape == (231, 1, 66) and a["joints"].shape == (231, 1, 22, 3)
    assert all(np.array_equal(a[n], b[n]) for n in a)
    np.testing.assert_allclose(a["poses"], golden("dance.npz")["poses"], rtol=0, atol=2e-5)


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
