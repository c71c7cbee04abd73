"""bench.py on the GPU: the default run prints one short, parseable result line, honours --steps, and --dump-outputs
writes the same outputs whatever the number of steps (the inputs are a fixed function of the arguments)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                         timeout=1800, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = out.stdout.splitlines()
    assert len(lines) == 1, out.stdout[:2000]
    return lines[0], out.stderr


def load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_default_bench_line_and_dumped_outputs(pkg, oracle, tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    text, err = run_bench("--gpus", "1", "--steps", "2", "--warmup", "1", "--dump-outputs", str(a))
    assert len(text) < 8192, len(text)           # the whole line must survive a reader that keeps the output's tail
    line = json.loads(text)
    assert line["steps"] == 2 and line["value"] > 0 and line["e2e"]["value"] > 0
    assert line["roofline"]["timing"]["step_units_per_step"] > 0
    detail = json.loads(err.strip().splitlines()[-1])["detail"]
    assert "config_C5_gallager100k_1M" in detail and "sweep" in detail

    z = load_dump(a)
    assert set(z) == {"syndrome_index", "errors", "converged", "iterations", "counters"}
    assert all(v.dtype in (np.float32, np.float64) for v in z.values())
    assert sum(os.path.getsize(os.path.join(a, f)) for f in os.listdir(a)) <= 64 << 20
    H, _, _ = pkg.codes.config_matrix("C3")
    k = len(z["syndrome_index"])
    assert z["errors"].shape == (k, H.shape[1]) and z["converged"].shape == z["iterations"].shape == (k,)
    assert z["counters"][0] == line["config"]["batch_per_gpu"]
    assert z["counters"][1] / z["counters"][0] == pytest.approx(line["converged_frac"])
    # a decoded error flagged converged reproduces its syndrome, regenerated from the bench's Philox stream
    for c in np.flatnonzero(z["converged"] == 1)[:64]:
        _, syn = oracle.sample(H, line["config"]["per"], 12345, int(z["syndrome_index"][c]), 1)
        assert np.array_equal((H @ z["errors"][c].astype(np.int64)) % 2, syn[:, 0].astype(np.int64))

    run_bench("--gpus", "1", "--steps", "1", "--warmup", "0", "--no-sweep", "--no-cpu", "--no-e2e", "--dump-outputs", str(b))
    zb = load_dump(b)
    for name in z:
        assert np.array_equal(z[name], zb[name]), name
