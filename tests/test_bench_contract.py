"""bench.py contract: the reference arm prints one JSON line with the agreed keys, the b200 arm refuses to run without a
GPU instead of falling back to anything, and on a GPU it dumps what its last timed step computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PERCENTILES = [0.0, 0.5, 0.75, 0.9, 0.95, 0.99, 0.999, 0.9999, 1.0]   # bench.py's


@pytest.mark.timeout(180)
def test_reference_arm_prints_contract_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=170, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "samples/s" and line["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["dtype"] == "f64" and line["data"] == "synthetic" and line["value"] > 1e5
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_dump_outputs_hold_the_last_timed_step(tmp_path, oracle):
    """--dump-outputs writes the reduction the last timed step returned: the oracle's reduction of the same seeded batch
    (stream U, indices [0, n)), whatever the number of steps.  The launch count shows --steps sets the timed steps."""
    import numpy as np
    n = 1_000_003
    runs = {}
    for steps in (1, 3):
        out = tmp_path / ("steps%d" % steps)
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--n", str(n),
                              "--no-e2e", "--no-api", "--no-cpu-baseline", "--sustain-seconds", "0", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=280, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["parity"]["ok"]
        files = sorted(out.iterdir())
        assert [f.name for f in files] == ["avgs.npy", "counts.npy", "pkeys.npy", "pvals.npy", "sums.npy"]
        assert sum(f.stat().st_size for f in files) <= 64 << 20
        runs[steps] = (line, {f.stem: np.load(f) for f in files})
    assert runs[3][0]["gpu_launches"] == 3 * runs[1][0]["gpu_launches"]
    ref = oracle.process_histogram(oracle.stream_ingest(oracle.STREAM_U, n, oracle.DEFAULT_SEED), PERCENTILES)
    for _, d in runs.values():
        assert all(v.dtype == np.float64 for v in d.values())
        assert d["counts"].tolist() == [n]
        assert (d["pkeys"][0] == ref["pkeys"]).all()
        assert (d["pvals"][0].view(np.uint64) == ref["pvals"].view(np.uint64)).all()
        assert abs(d["sums"][0] - ref["sum"]) <= 1e-12 * abs(ref["sum"])
        assert abs(d["avgs"][0] - ref["avg"]) <= 1e-12 * abs(ref["avg"])


def test_b200_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=170, cwd=ROOT)
    assert res.returncode != 0
    assert "no CPU fallback" in (res.stderr + res.stdout)
