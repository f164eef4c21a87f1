"""bench.py --dump-outputs on the device: the files hold what the public solveBatch returns on the workload's seeded
inputs, and the run prints its one JSON line as usual."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_outputs_match_solve_batch(tmp_path):
    import icnn_b200
    from icnn_b200 import bundle_entropy, workloads
    d = tmp_path / "out"
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", "2",
                          "--warmup", "1", "--no-sub", "--no-cpu-baseline", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert run.returncode == 0, run.stderr[-2000:]
    lines = [l for l in run.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    out = {f[:-4]: np.load(str(d / f)) for f in os.listdir(str(d))}
    assert sum(a.nbytes for a in out.values()) <= 64 << 20

    cfg = workloads.CONFIGS["C1"]
    p, x, y0 = workloads.make_inputs("C1")
    net = icnn_b200.PICNN.from_params(p, device="cuda:0")
    y, A, b, lam, xs, nIters = bundle_entropy.solveBatch(net.bind(x, affine=cfg["affine"]), y0.copy(),
                                                         nIter=cfg["nIter"])
    rows = out["row_index"].astype(int)
    assert len(rows) == cfg["B"]                 # C1 is small enough to be written whole
    np.testing.assert_allclose(out["x"], y[rows], rtol=0, atol=1e-12)
    np.testing.assert_array_equal(out["nIters"], np.array(nIters)[rows])
    np.testing.assert_array_equal(out["counts"], [len(A[u]) for u in rows])
    for i, u in enumerate(out["bundle_row_index"].astype(int)):
        k = len(A[u])
        np.testing.assert_allclose(out["A"][i, :k], np.array(A[u]).reshape(k, -1), rtol=0, atol=1e-6)
        np.testing.assert_allclose(out["xs"][i, :k], np.array(xs[u]).reshape(k, -1), rtol=0, atol=1e-12)
        np.testing.assert_allclose(out["b"][i, :k], b[u], rtol=0, atol=1e-12)
        if k:
            np.testing.assert_allclose(out["lam"][i, :k], lam[u], rtol=0, atol=1e-12)
