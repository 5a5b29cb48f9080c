"""GPU: bench.py --dump-outputs writes what the timed path returned in its last step, so that two builds can be compared
output for output on the benchmark's own seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("theta", "fpkm", "frac", "tpm", "keep", "iters", "status")


def test_dump_outputs_equal_a_plain_solve_of_the_benchmark_batch(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0", "--no-giant",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and "error" not in line["bias"]
    files = {p.name: np.load(p) for p in tmp_path.iterdir()}
    assert set(files) == {f"{p}{k}.npy" for p in ("", "bias_") for k in KEYS} | {"bias_beta.npy", "bias_outer.npy"}
    assert all(a.dtype == np.float64 for a in files.values())
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    from strawberry_b200 import api, synth
    b = synth.human_shaped(seed=2)
    q = api.Quantifier()
    q.submit_flat(b)
    q.run(b["total_mapped_reads"])
    ref = q.results()
    q.close()
    for k in KEYS:
        assert np.array_equal(files[f"{k}.npy"], ref[k].astype(np.float64), equal_nan=True), k
        assert files[f"bias_{k}.npy"].shape == ref[k].shape, k
    assert files["bias_beta.npy"].shape == (len(ref["status"]), 5)
