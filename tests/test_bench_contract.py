"""bench.py's reference arm on the CPU: one JSON line with the contract's keys (the GPU arm needs a device and is run by the driver)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-chunks", "2"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "MB/s" and d["higher_is_better"] is True and d["value"] > 0
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_refuses_arguments_it_cannot_honour(argv, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120, cwd=tmp_path)
    assert out.returncode == 2 and "error:" in out.stderr, out.stderr[-2000:]
    assert not out.stdout.strip() and not os.listdir(tmp_path)
