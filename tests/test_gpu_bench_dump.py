"""bench.py --dump-outputs: what the timed step returned, in a form two builds can be compared with."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_are_the_propagated_table_and_reproducible(tmp_path):
    # scale 0.001: 10 000 users x 5 000 items, N = 15 001 rows < DUMP_ROWS, so the sample is the whole table
    cmd = [sys.executable, "bench.py", "--scale", "0.001", "--steps", "3", "--warmup", "1", "--no-train", "--no-eval",
           "--no-e2e", "--no-small-configs", "--no-cpu-baseline"]
    runs = []
    for k in range(2):
        out = subprocess.run(cmd + ["--dump-outputs", str(tmp_path / str(k))], cwd=ROOT, capture_output=True,
                             text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
        runs.append({f[:-4]: np.load(tmp_path / str(k) / f) for f in os.listdir(tmp_path / str(k))})
    a, b = runs
    assert set(a) == {"propagated_sample", "propagated_sample_rows", "propagated_col_sum"}
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    N = 10_000 + 1 + 5_000
    assert np.array_equal(a["propagated_sample_rows"], np.arange(N, dtype=np.float64))
    assert a["propagated_sample"].shape == (N, 64) and a["propagated_col_sum"].shape == (64,)
    assert np.allclose(a["propagated_sample"].astype(np.float64).sum(0), a["propagated_col_sum"], rtol=1e-9, atol=1e-9)
    # seeded inputs, no atomics in the propagation: the same bits on every run
    assert np.array_equal(a["propagated_sample"], b["propagated_sample"])
    assert np.allclose(a["propagated_col_sum"], b["propagated_col_sum"], rtol=1e-12, atol=0)
