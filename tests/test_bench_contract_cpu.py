"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) runs the CPU port
on this host and prints ONE JSON line with the keys the driver reads; the CUDA arm fails loudly
without a device instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C1",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["higher_is_better"] is True
    assert d["unit"] == "solves/s" and d["value"] > 0 and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] and "workload" in d["config"]
    # the reference arm maps no native code: icnn_b200's package init is lazy and bench.py only touches
    # icnn_b200.workloads (pure numpy) on this arm (VERDICT r01, measurement hygiene 7)
    assert d["native_modules_loaded"] == []
    assert d["config"]["workload"].startswith("C1: ") and "/GPU" not in d["config"]["workload"]


def test_workloads_import_does_not_load_the_native_library():
    code = ("import sys; from icnn_b200 import workloads; "
            "assert 'icnn_b200._capi' not in sys.modules and 'torch' not in sys.modules; print('ok')")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-1000:]


def test_default_workload_is_the_largest_single_gpu_config():
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'ap.add_argument("--workload", default="C5"' in src
    assert 'scaling = args.scaling or "strong"' in src


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_cuda_arm_fails_loudly_without_a_gpu():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", "1",
                          "--warmup", "1", "--no-cpu-baseline"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert not [l for l in out.stdout.splitlines() if l.startswith("{")]      # no number without a device


def test_reference_arm_under_torchrun_prints_one_line_from_rank_0():
    """The driver launches the reference arm like the CUDA arm at N > 1 (torchrun, one rank per GPU): rank 0 alone
    runs the CPU path and prints the line, the other ranks exit 0 without work."""
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "bench.py"),
                          "--impl", "reference", "--gpus", "2", "--workload", "C1", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0 and d["native_modules_loaded"] == []


def _load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_writes_the_ragged_results_of_sampled_rows(tmp_path, monkeypatch):
    """--dump-outputs: the arrays solveBatch returns for a fixed row sample, bundle rows in perm order (what the
    ragged A / b / lam / xs views hold), zero past counts, float32 / float64 only, within the 64 MB budget."""
    import types
    import numpy as np
    bench = _load_bench()
    assert bench.DUMP_X_BYTES + bench.DUMP_BUNDLE_BYTES + 16 * 1024 <= 64 << 20
    B, n, KS = 9, 5, 4
    g = torch.Generator().manual_seed(0)
    st = types.SimpleNamespace(
        B=B, n=n, KS=KS, y=torch.rand(B, n, generator=g, dtype=torch.float64),
        G=torch.randn(B, KS, n, generator=g), ys=torch.rand(B, KS, n, generator=g, dtype=torch.float64),
        h=torch.randn(B, KS, generator=g, dtype=torch.float64), lam=torch.rand(B, KS, generator=g, dtype=torch.float64),
        perm=torch.stack([torch.randperm(KS, generator=g) for _ in range(B)]).int(),
        count=torch.randint(0, KS + 1, (B,), generator=g).int(), nIters=torch.randint(1, 6, (B,), generator=g).int())
    monkeypatch.setattr(bench, "DUMP_X_BYTES", 6 * (8 * n + 24))                # 6 of 9 rows
    monkeypatch.setattr(bench, "DUMP_BUNDLE_BYTES", 4 * (KS * (12 * n + 16) + 8))  # 4 of those 6
    runs = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), st)
        runs.append({f[:-4]: np.load(str(tmp_path / d / f)) for f in os.listdir(str(tmp_path / d))})
    out = runs[0]
    assert sorted(out) == ["A", "b", "bundle_row_index", "counts", "lam", "nIters", "row_index", "x", "xs"]
    for k, a in out.items():
        assert a.dtype in (np.float32, np.float64), k
        np.testing.assert_array_equal(a, runs[1][k], err_msg=k)       # same state -> same sample, same files
    rows, brows = out["row_index"].astype(int), out["bundle_row_index"].astype(int)
    assert len(rows) == 6 and len(set(rows)) == 6 and len(brows) == 4 and set(brows) <= set(rows)
    np.testing.assert_array_equal(out["x"], st.y.numpy()[rows])
    np.testing.assert_array_equal(out["nIters"], st.nIters.numpy()[rows])
    np.testing.assert_array_equal(out["counts"], st.count.numpy()[rows])
    assert out["A"].dtype == np.float32 and out["A"].shape == (4, KS, n) and out["xs"].shape == (4, KS, n)
    for i, u in enumerate(brows):
        k = int(st.count[u])
        slots = st.perm.numpy()[u, :k]
        for name, src in (("A", st.G), ("xs", st.ys), ("b", st.h), ("lam", st.lam)):
            np.testing.assert_array_equal(out[name][i, :k], src.numpy()[u, slots], err_msg=name)
            assert not np.any(out[name][i, k:]), name


def test_algorithmic_work_models_match_survey_8d():
    """The roofline numerators: FLOP_fg = 4 * MAC per solve (SURVEY.md 8d: C2 9.45 M, C3 0.866 M, C4 0.170 M,
    C5 79.7 M, T 8.39 M) and the K2 FP64 model n (k^2 + 11 k + 30) per interior-point iteration (DESIGN.md section 3)."""
    import numpy as np
    bench = _load_bench()
    from icnn_b200 import workloads
    want = {"C1": 4 * 536, "C2": 4 * 2361856, "C3": 4 * 216399, "C4": 4 * 42606, "C5": 4 * 19928064, "T": 4 * 2098688}
    for name, flops in want.items():
        assert bench.flop_fg(workloads.CONFIGS[name]) == float(flops), name
    # one sample, one iteration entered, 3 interior-point iterations with k = 5 rows, n = 100
    stats = np.zeros((1, 8))
    stats[0, 2], stats[0, 3], stats[0, 4] = 3, 3 * 25, 3 * 5
    assert bench.k2_fp64_flops(100, stats) == 100.0 * 3 * (25 + 55 + 30)
    assert bench.workload_string("T", workloads.CONFIGS["T"]).startswith("T: m=512 n_y=512 hidden=[1024, 1024] batch=4096 nIter=10")
