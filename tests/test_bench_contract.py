"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`, the unmodified reference
package installed in oracle/_ref by build(), on the host cores; the oracle port when none is installed) must print
ONE JSON line carrying the same metric / unit / workload as the GPU arm plus the keys its readers use; ranks other
than 0 print nothing; --steps below 1 is refused."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def _run(env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    return [ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")]


def test_reference_arm_json_line():
    sys.path.insert(0, ROOT)
    import bench
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["workload"] == bench.workload_name()
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if bench.reference_available() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "rows" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_rank0_only():
    assert _run({"RANK": "1", "WORLD_SIZE": "2"}) == []


def test_steps_below_one_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr
