"""bench.py's CPU arm prints the one JSON line of the contract (no GPU needed for --impl reference); on the GPU, the
outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "leduc_pot",
                          "--steps", "3", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in d["config"]


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_fhp_steps(tmp_path):
    """--dump-outputs writes float arrays within 64 MB; the trace covers exactly --steps iterations, and a second run with
    the same arguments writes the same outputs bit for bit."""
    dumps = []
    for run in range(2):
        d_out = tmp_path / ("run%d" % run)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--fhp-boards", "512", "--steps", "40",
                              "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(d_out)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 40
        dumps.append({p.stem: np.load(p) for p in sorted(d_out.glob("*.npy"))})
    a, b = dumps
    assert set(a) == {"exploitability", "regret_rows", "avg_rows", "trunk_regret", "trunk_strat", "trunk_avg"}
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert a["exploitability"][:, 0].tolist() == [20, 40]
    assert a["regret_rows"].shape[:2] == (256, 14) and np.any(a["regret_rows"] != 0)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
