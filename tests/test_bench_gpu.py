"""GPU test of bench.py's engine arm: `--steps` sets the number of timed steps, and `--dump-outputs` writes the C of
the last timed step (config 1 is small enough to be written whole) as the host oracle computes it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_is_the_product(tmp_path):
    from oracle import host
    from pem_spgemm_b200 import synth
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--steps", "2", "--warmup", "3",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == line["e2e"]["steps"] == line["e2e_coo"]["steps"] == 2
    got = {k: np.load(tmp_path / f"{k}.npy") for k in ("C_nnz", "C_rows", "C_cols", "C_vals")}
    assert all(a.dtype == np.float64 for a in got.values())
    _, _, C = host.spgemm_from_coo(*synth.laplacian2d(256), False)
    r, c, v = C.to_coo()
    assert got["C_nnz"].tolist() == [C.nnz] == [line["workload_stats"]["nnz_C"]]
    assert np.array_equal(got["C_rows"], r) and np.array_equal(got["C_cols"], c) and np.array_equal(got["C_vals"], v)
