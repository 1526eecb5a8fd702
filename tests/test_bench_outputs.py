"""bench.py --dump-outputs: the headline arm's last timed step, as float64 arrays, equals the oracle's bindings."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from yunikorn_k8shim_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_are_the_oracle_bindings(oracle, tmp_path):
    out = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--quick", "--steps", "2", "--warmup", "3",
                        "--dump-outputs", str(out)], capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["steps"] == 2 and res["bindings_identical_to_oracle"]
    want = oracle.run(synth.perf())                       # the default workload, config 2
    for name in ("ask", "node"):
        got = np.load(out / f"{name}.npy")
        assert got.dtype == np.float64
        assert np.array_equal(got, want[name].astype(np.float64)), name
