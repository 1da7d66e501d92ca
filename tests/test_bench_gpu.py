"""bench.py's own arm on the GPU: one JSON line for the requested number of timed steps, and --dump-outputs writes
what the last timed step (the replayed CUDA-graph step) computed -- the same, up to rounding, in every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from test_bench_cpu import check_dumped_outputs

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "3",
                          "--batch", "8", "--no-cpu-baseline", "--no-variants", "--no-gpu-reference",
                          "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-4000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_bench_dumps_the_last_timed_step_the_same_in_every_run(tmp_path):
    runs = [tmp_path / "a", tmp_path / "b"]
    for run in runs:
        d = _bench(run)
        assert d["steps"] == 3 and d["value"] > 0 and d["config"]["batch_per_gpu"] == 8
        assert d["config"]["launch"].startswith("whole training step replayed as one CUDA graph")
        check_dumped_outputs(run)
    # the dumped step starts from the seeded initial state: two runs differ only by the summation order of the
    # atomics within that one step
    for p in sorted(runs[0].iterdir()):
        a, b = float(np.load(p)), float(np.load(runs[1] / p.name))
        assert abs(a - b) <= 1e-3 * abs(a), (p.name, a, b)
