"""bench.py prints exactly ONE JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def run_bench(*args, timeout):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, f"stdout must be one JSON line, got {len(lines)}"
    return json.loads(lines[0])


def test_reference_arm_line():
    """`--impl reference`: the unmodified reference learner (oracle/_ref or /root/reference; the
    float64 port only where neither exists) on the same workload, here the small c3 config."""
    from oracle import refload

    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "1", "--config", "c3", timeout=600)
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "steps/s"
    assert d["value"] > 0 and d["steps"] == 1 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if refload.available() else "port")
    assert cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["config"]["B"] == 1024 and d["config"]["global_batch"] == 1024
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 == d["e2e"]["d2h_bytes_per_step"]


@pytest.mark.gpu
def test_own_arm_line(tmp_path):
    """Default arm on cuda:0: contract keys, a dominant-kernel roofline, clocks, launch count, and the
    outputs of the last timed step under --dump-outputs."""
    import numpy as np

    d = run_bench("--steps", "5", "--warmup", "3", "--no-cpu", "--dump-outputs", str(tmp_path / "out"), timeout=600)
    dumped = {f[:-4]: np.load(tmp_path / "out" / f) for f in os.listdir(tmp_path / "out")}
    assert {"scalars", "vs", "pg_adv", "params.policy.model.0.weight", "grad.value_fn.model.3.bias"} <= set(dumped)
    assert all(a.dtype in (np.float32, np.float64) for a in dumped.values())
    assert sum(a.nbytes for a in dumped.values()) <= 64 << 20
    assert dumped["scalars"][3] == d["loss"]["device_resident"]
    assert dumped["vs"].shape == (d["config"]["T"] + 1, d["config"]["B"]) and np.isfinite(dumped["vs"]).all()
    assert (BASE_KEYS - {"cpu_baseline"}) | {"roofline", "clocks", "gpu_launches", "kernels"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["warmup"] >= 3 and d["value"] > 0
    assert abs(d["value"] * d["ms_per_step"] - 1e3) < 1e-6 * 1e3
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    assert d["gpu_launches"] >= 3 * d["steps"]
    assert d["clocks"]["sm_max_mhz"] > 0 and d["clocks"]["sm_mhz"] > 0 and isinstance(d["clocks"]["reasons"], list)
    assert sum(1 for k in d["kernels"].values() if k.get("in_step")) >= 3
    par = d["parity"]  # first step of this configuration against the float64 oracle (oracle/check.py)
    assert par["ok"] and par["max_abs_vs"] < 1e-5 and par["max_abs_pg"] < 1e-5 and par["max_abs_scalar"] < 1e-5, par
