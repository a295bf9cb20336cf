"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) runs the reference's own
SimclrLoss (staged copy in baseline/_ref, else /root/reference; the oracle port when neither exists) on a bounded
sample and prints ONE JSON line with the keys the driver reads; under torchrun only rank 0 works."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_json_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ntxent_fwd_bwd_samples_per_s" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["config"]["global_batch"] == 32768 and d["config"]["dim"] == 128
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    if cb["kind"] == "reference":   # the reference's classes cannot run N = 32768: the sample size and the N^2 law are stated
        assert cb["extrapolated"] is True and "utils/losses.py:8-46" in cb["sample"] and "extrapolated" in cb["sample"]
    else:
        assert "row slab" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    assert _run({"RANK": "3", "WORLD_SIZE": "8", "LOCAL_RANK": "3"}) == []


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "DIR"]])
def test_bad_arguments_are_refused(tmp_path, extra):
    """No timed step means no time, and --dump-outputs writes what the CUDA path returns, so both are usage errors."""
    args = [a.replace("DIR", str(tmp_path / "out")) for a in extra]
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "error:" in out.stderr
    assert not (tmp_path / "out").exists()


def test_reference_arm_falls_back_to_port_without_reference(tmp_path):
    """On a box with neither baseline/_ref nor /root/reference the arm still runs (oracle port) and says so."""
    code = ("import sys, types; sys.argv=['bench.py','--impl','reference','--steps','1','--warmup','0'];"
            "import oracle.ref_loader as rl; rl.find_root=lambda: None;"
            "import runpy; runpy.run_path('bench.py', run_name='__main__')")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["cpu_baseline"]["kind"] == "port" and "row slab" in d["cpu_baseline"]["sample"]
