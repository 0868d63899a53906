"""bench.py on the GPU: --steps and --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_repeat_from_run_to_run(tmp_path):
    """Two runs with the same arguments dump the same detections: the inputs are seeded, so two builds can be compared."""
    dumps = []
    for run in ("a", "b"):
        args = ["--steps", "3", "--warmup", "1", "--batch", "2", "--no-cpu", "--no-clip", "--dump-outputs", str(tmp_path / run)]
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 3
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("detections", "e2e_detections", "head")})
    for n, a in dumps[0].items():
        assert a.shape[:2] == ((2, 84) if n == "head" else (2, 300)) and a.dtype == np.float32 and np.isfinite(a).all(), n
        np.testing.assert_array_equal(a, dumps[1][n], err_msg=n)
    assert dumps[0]["head"][:, 4:].max() > 0                         # class probabilities: not an empty buffer
