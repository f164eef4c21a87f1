#!/usr/bin/env python
"""bench.py -- inner-loop solves/sec of the ICNN argmin path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C5] [--scaling strong|weak] [--impl reference]

One "step" = one solveBatch over one minibatch of synthetic input.  Headline workload (default) = C5 =
BASELINE.json configs[4], the largest single-GPU configuration (n_y=4096, 4x1024 hidden, batch 8192,
50 bundle iterations); with --gpus N the batch is SHARDED over the ranks by default (strong scaling,
lib/bundle_entropy.py:211: samples are independent), one all-gather of y* at the end.
metric = B x iterations-executed / seconds ("a solve" = one sample advanced one inner iteration;
iterations-executed honours the reference's early return, lib/bundle_entropy.py:239).  Prints ONE JSON line.

  value        device-resident: gates + y0 already in HBM, CUDA-event time of the fused loop
  e2e          same metric through the public API with HOST buffers (icnn_b200.bundle_entropy.solveBatch /
               icnn_b200.dist.solve_batch_sharded: H2D of x and y0, x-path gate GEMMs, loop, D2H of y*)
  roofline     dominant kernel class: CUDA-event time from an instrumented pass, algorithmic work from the
               per-iteration statistics the kernels accumulate (DESIGN.md section 3), measured peaks
  cpu_baseline the numpy oracle port of the reference's solveBatch on the host cores (bounded sample) and the
               reference's own cost model (dense np.diag, prints, one thread) on a tiny sample
  configs      sub-records (N=1 only) for the other BASELINE.json configs and the north-star target shape:
               T (batch 4096 / n_y 512), C2 (Olivetti dims), C3 (Bibtex dims: bundle AND 30-step GD), C4 (RL dims),
               each with its own value / e2e / roofline / cpu_baseline

--impl reference: times the CPU implementation only (oracle port; the reference itself is Python and
/root/reference does not exist on the GPU box), all host cores, same metric/config; loads no native code.

--dump-outputs DIR: after the timed steps of the headline workload, write what its last step returned (y*, the
bundle, nIters; see dump_outputs) as DIR/<name>.npy, so that two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "inner-loop solves/sec (batch x iters)"
UNIT = "solves/s"
SUB_WORKLOADS = ["T", "C2", "C3", "C4"]


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return dict(hbm_gbs=float(pk["hbm_gbs"]), bf16_tflops=float(pk["bf16_tflops"]),
                    bf16_sustained=float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"])),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0,
                source="fallback (B200_PROFILING.md)")


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` captures (profiles/r02_traffic.json: {workload: {kernel, t, bytes, source}})."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


def workload_string(name, cfg, solver="pc"):
    return ("%s: m=%d n_y=%d hidden=%s batch=%d nIter=%d variant=%s solver=%s"
            % (name, cfg["m"], cfg["n"], cfg["hidden"], cfg["B"], cfg["nIter"], cfg["variant"], solver))


def flop_fg(cfg):
    """Algorithmic FLOPs of one f/grad row (SURVEY.md 8d): 4 * (n * sum s_i + sum s_{i-1} s_i)."""
    s = list(cfg["hidden"]) + [1]
    mac = cfg["n"] * sum(s) + sum(s[i - 1] * s[i] for i in range(1, len(s)))
    return 4.0 * mac


def k2_fp64_flops(n, stats):
    """Algorithmic FP64 FLOPs of the per-sample solves of one solveBatch (DESIGN.md section 3, K2): per
    interior-point / Newton iteration of a sample with k active rows
        2 n (k(k+1)/2 + 2k)   weighted Gram G D G^T + the two products G(D ry), G y
      + 2 n 3k                G^T [dz_aff dz_p dz_q]
      + 30 n                  elementwise (D, dy, du, updates, step bounds; log / division internals not counted)
      = n (k^2 + 11 k + 30);  the k x k factor / solves (k^3/3 + 8 k^2) are left out (< 2 %).
    stats = per-iteration totals (icnn_bundle_bufs::iter_stats): [3] = sum its*k^2, [4] = sum its*k, [2] = sum its."""
    return float(n) * float(stats[:, 3].sum() + 11.0 * stats[:, 4].sum() + 30.0 * stats[:, 2].sum())


# ------------------------------------------------------------------------------------------
# CPU side (oracle port) -- the only place bench.py executes oracle/
# ------------------------------------------------------------------------------------------

_WORKER_CACHE = {}      # one entry per worker process: (workload, seed, Bgen) -> (p, x, y0)


def _cpu_worker(args):
    workload, seed, lo, hi, Bgen, nIter, dense_diag, verbose = args
    from threadpoolctl import threadpool_limits
    from oracle import bundle_np, picnn_np
    from icnn_b200 import workloads
    cfg = workloads.CONFIGS[workload]
    key = (workload, seed, Bgen)
    if key not in _WORKER_CACHE:      # the pool's processes persist across steps: generate theta / inputs once (untimed
        _WORKER_CACHE.clear()         # either way; at C5 it is 3 s and 0.4 GB per process), keep only the latest
        _WORKER_CACHE[key] = workloads.make_inputs(workload, B=Bgen, seed=seed)
    p, x, y0 = _WORKER_CACHE[key]
    x, y0 = x[lo:hi], y0[lo:hi].copy()
    # float32 arithmetic mimics the reference's TF-backed fg; the values are handed over in float64
    # arrays so that the CPU arm does the same work as the GPU arm: np.linalg.matrix_rank scales its
    # tolerance with the row dtype, and with float32-typed rows most samples hit the rank stop early
    # (they would still be counted as "solves" while doing nothing)
    fg = picnn_np.make_fg(p, x, dtype=np.float32, out_dtype=np.float64, affine=cfg["affine"])
    iters = [0]

    def cb(t, *a):
        iters[0] = t + 1

    kw = {}
    if dense_diag:
        kw["dense_diag"] = True
    if verbose:   # the reference prints one line per interior-point iteration (lib/bundle_entropy.py:34-36)
        kw["verbose"] = True
        sys.stdout = open(os.devnull, "w")
    with threadpool_limits(limits=1), np.errstate(all="ignore"):
        t0 = time.perf_counter()
        bundle_np.solve_batch(fg, y0, nIter=nIter, variant=cfg["variant"], callback=cb, **kw)
        dt = time.perf_counter() - t0
    if verbose:
        sys.stdout = sys.__stdout__
    return (hi - lo) * iters[0], dt


def usable_cores():
    """Host cores this process may really use: min(affinity mask, cgroup v2/v1 CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path, parse in (("/sys/fs/cgroup/cpu.max", lambda t: t.split()),
                        ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", lambda t: [t.strip(), open(
                            "/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().strip()])):
        try:
            q, per = parse(open(path).read())
            if q != "max" and int(q) > 0:
                n = min(n, max(1, int(int(q) / int(per))))
            break
        except Exception:
            continue
    return max(1, n)


_POOL = {}


def _close_pools():
    for pl in _POOL.values():
        pl.terminate()
        pl.join()
    _POOL.clear()


def _noop(_):
    return 0


def _pool(procs):
    import multiprocessing as mp
    if procs not in _POOL:
        # spawn (not fork): the parent may hold an initialised CUDA context and torch threads
        _POOL[procs] = mp.get_context("spawn").Pool(procs)
        _POOL[procs].map(_noop, range(procs * 2))     # start every worker before anything is timed
    return _POOL[procs]


def cpu_reference(workload, rows, procs, seed=None, nIter=None, dense_diag=False, verbose=False):
    """Oracle-port solveBatch on ``rows`` rows of the workload, split over ``procs`` processes
    (samples are independent, lib/bundle_entropy.py:211).  Returns (solves, seconds) where
    seconds = the slowest worker's solveBatch time (process start-up / input generation not counted)."""
    from icnn_b200 import workloads
    cfg = workloads.CONFIGS[workload]
    nIter = cfg["nIter"] if nIter is None else nIter
    seed = cfg["seed"] if seed is None else seed
    rows = max(1, min(rows, cfg["B"]))
    procs = max(1, min(procs, rows))
    bounds = [(rows * i) // procs for i in range(procs + 1)]
    jobs = [(workload, seed, bounds[i], bounds[i + 1], rows, nIter, dense_diag, verbose) for i in range(procs)]
    res = _pool(procs).map(_cpu_worker, jobs, chunksize=1)
    return sum(r[0] for r in res), max(r[1] for r in res)


def cpu_plan(workload, procs, budget_s):
    """(rows, nIter) of a bounded sample: calibrate on one row per process for min(nIter, 6) iterations (the cost
    of an iteration grows with the bundle, ~ quadratic cumulative cost), then take the full iteration count if
    one row per process fits the budget, else the largest iteration count that does (the first, CHEAPEST
    iterations -- an upper bound of the CPU throughput, i.e. conservative for the GPU/CPU ratio)."""
    from icnn_b200 import workloads
    cfg = workloads.CONFIGS[workload]
    nfull = cfg["nIter"]
    ncal = min(nfull, 6)
    cal_rows = min(cfg["B"], procs)
    _s, w = cpu_reference(workload, cal_rows, procs, nIter=ncal)
    expo = 1.5     # measured: cumulative cost of t iterations ~ t^1.5 (the bundle grows, pruning keeps k << t)
    est_full = w * (nfull / float(ncal)) ** expo
    if est_full > budget_s and ncal < nfull:
        # second calibration point closer to the budget before giving up on the full iteration count
        n2 = min(nfull, max(ncal + 1, int(ncal * (budget_s / max(w, 1e-3)) ** (1.0 / expo))))
        _s, w2 = cpu_reference(workload, cal_rows, procs, nIter=n2)
        est_full = w2 * (nfull / float(n2)) ** expo
        ncal, w = n2, w2
    if est_full <= budget_s:
        rows_per_proc = max(1, int(budget_s / max(est_full, 1e-3)))
        return min(cfg["B"], procs * rows_per_proc), nfull, w
    its = max(1, min(nfull, int(ncal * (budget_s / max(w, 1e-3)) ** (1.0 / expo))))
    return cal_rows, its, w


def cpu_baseline(workload, budget_s=15.0, reference_cost=False):
    """Bounded sample sized for ~budget_s seconds on all host cores."""
    from icnn_b200 import workloads
    cfg = workloads.CONFIGS[workload]
    procs = usable_cores()
    rows, its, _ = cpu_plan(workload, procs, budget_s)
    solves, wall = cpu_reference(workload, rows, procs, nIter=its)
    out = dict(value=solves / wall, unit=UNIT, cores=min(procs, rows), kind="port",
               sample="%d of %d rows x %d of %d iterations (%d solves executed, %.1f s wall), numpy oracle port of "
                      "lib/bundle_entropy.solveBatch(solver='pc') / the RL copy for C4, float32-arithmetic fg, "
                      "%d processes x 1 BLAS thread" % (rows, cfg["B"], its, cfg["nIter"], solves, wall,
                                                        min(procs, rows)))
    if reference_cost and cfg["variant"] == "lib":
        # the reference's own cost model: dense np.diag n x n matrices (lib/bundle_entropy.py:17-18,41), one line
        # printed per interior-point iteration (:34-36), one Python thread -- BASELINE.md section 3
        its_rc = min(cfg["nIter"], 3 if cfg["n"] > 1024 else 5)
        s_rc, w_rc = cpu_reference(workload, 1, 1, nIter=its_rc, dense_diag=True, verbose=True)
        out["reference_cost"] = dict(
            value=s_rc / w_rc, unit=UNIT, cores=1,
            sample="1 row x %d iterations (%.1f s), the port with the reference's dense np.diag hess/hess_inv "
                   "matrices and per-iteration prints (stdout discarded), one process x 1 BLAS thread" % (its_rc, w_rc))
    return out


# ------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.reasons, self.max = index, [], set(), None
        self._stop = threading.Event()
        self._th = None

    def _run(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._th.join(timeout=6)

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        return dict(sm_mhz=med, sm_max_mhz=self.max, reasons=sorted(self.reasons), samples=len(self.samples))


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------

class Ctx:
    pass


def measure_fp64_peak(ctx):
    """FP64 tensor-core (DMMA m8n8k4) throughput of this GPU, measured live: the denominator of K2's roofline
    (MEASURED_PEAKS.json carries HBM and bf16 only)."""
    import ctypes as C
    import torch
    from icnn_b200 import _capi
    out = torch.zeros(1, dtype=torch.float64, device=ctx.dev)
    iters = 4096
    flops = C.c_double(0.0)
    best = 0.0
    for rep in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _capi.check(_capi.lib.icnn_fp64_mma_probe(iters, out.data_ptr(), C.byref(flops), ctx.stream))
        e1.record()
        torch.cuda.synchronize()
        if rep:
            best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


DUMP_X_BYTES = 32 << 20         # --dump-outputs: y* rows and their per-row scalars
DUMP_BUNDLE_BYTES = 24 << 20    # --dump-outputs: bundle rows (A in float32 + xs in float64, KS x n each; b, lam)


def dump_outputs(out_dir, st):
    """Write what solveBatch returns, (x, A, b, lam, xs, nIters), for a fixed sample of rows of ``st`` as
    out_dir/<name>.npy: x [R, n] and nIters / counts [R] for R rows (all rows when they fit DUMP_X_BYTES, else a
    sample drawn with a fixed seed), A / xs [R', KS, n] and b / lam [R', KS] for R' of those rows spread evenly
    (DUMP_BUNDLE_BYTES), in bundle order (A[u][j] = the reference's ragged A[u][j]), zero past counts; row_index /
    bundle_row_index give the rows.  Every array is float32 or float64; the sample depends only on the shape."""
    import torch
    B, n, KS = st.B, st.n, st.KS
    nx = min(B, max(1, DUMP_X_BYTES // (8 * n + 3 * 8)))                   # x, nIters, counts, row_index
    nb = min(nx, max(1, DUMP_BUNDLE_BYTES // (KS * (12 * n + 16) + 8)))    # A, xs, b, lam, bundle_row_index
    rows = np.arange(B) if nx == B else np.sort(np.random.RandomState(0).choice(B, nx, replace=False))
    brows = rows[np.linspace(0, nx - 1, nb).round().astype(np.int64)]
    out = {"row_index": rows.astype(np.float64), "bundle_row_index": brows.astype(np.float64)}
    idx = torch.from_numpy(rows).to(st.y.device)
    out["x"] = st.y.index_select(0, idx).cpu().numpy()
    out["nIters"] = st.nIters.index_select(0, idx).cpu().numpy().astype(np.float64)
    out["counts"] = st.count.index_select(0, idx).cpu().numpy().astype(np.float64)
    bidx = torch.from_numpy(brows).to(st.y.device)
    perm = st.perm.index_select(0, bidx).long().clamp_(0, KS - 1)
    live = torch.arange(KS, device=perm.device)[None, :] < st.count.index_select(0, bidx)[:, None]
    for name, src in (("b", st.h), ("lam", st.lam)):
        out[name] = (src.index_select(0, bidx).gather(1, perm) * live).cpu().numpy()
    for name, src in (("A", st.G), ("xs", st.ys)):
        v = src.index_select(0, bidx).gather(1, perm[:, :, None].expand(-1, -1, n))
        out[name] = (v * live[:, :, None]).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_workload(ctx, name, steps, warmup, scaling, solver, cpu_seconds, headline, dump_dir=None):
    """value / e2e / per-kernel roofline / cpu_baseline of one workload on this rank set."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    import icnn_b200
    from icnn_b200 import _capi, bundle_entropy, workloads
    from icnn_b200 import dist as idist

    rank, world, dev, stream, flush = ctx.rank, ctx.world, ctx.dev, ctx.stream, ctx.flush
    cfg = workloads.CONFIGS[name]
    Bfull, n, nIter = cfg["B"], cfg["n"], cfg["nIter"]
    strong = (scaling == "strong")
    if strong:
        p, x_all, y0_all = workloads.make_inputs(name)
        lo, hi = idist.shard_rows(Bfull, rank, world)
        x, y0 = x_all[lo:hi], y0_all[lo:hi]
        Bglob, B = Bfull, hi - lo
    else:
        # weak scaling: every rank solves its own B rows (different seed -> different rows); theta = rank 0's
        p, x, y0 = workloads.make_inputs(name, seed=cfg["seed"] + 7919 * rank)
        if rank:
            p = workloads.make_inputs(name, B=1)[0]
        x_all, y0_all = x, y0
        Bglob, B = Bfull * world, Bfull
    net = icnn_b200.PICNN.from_params(p, device=dev)
    x_pin = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).pin_memory()
    y0_pin = torch.from_numpy(np.ascontiguousarray(y0)).pin_memory()
    variant = cfg["variant"]
    KS = (nIter if variant == "rl" else min(nIter, n)) + 1
    ccfg = bundle_entropy._make_cfg(variant, solver, nIter, None, None, 0, n, KS)
    y_all = torch.empty(Bglob, n, dtype=torch.float64, device=dev) if world > 1 else None

    def gather(y_local):
        if strong:
            y_all.copy_(idist.allgather_rows(y_local, Bglob))
        else:
            dist.all_gather_into_tensor(y_all, y_local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident step -----------------------------------------------------------------
    fg = net.bind(x_pin.to(dev), affine=cfg["affine"])
    st = bundle_entropy.BundleState(B, n, KS, dev, keep_xs=True, nIter=nIter, stats=True)
    stats_ptr = st.c.iter_stats
    st.c.iter_stats = None                      # statistics (atomics) only in the instrumented pass
    y0_dev = y0_pin.to(dev)

    def step_device():
        st.y.copy_(y0_dev)
        _capi.check(_capi.lib.icnn_solve_batch_fused(net._h, C.byref(fg.c_gates), C.byref(ccfg), C.byref(st.c),
                                                     fg.ws.data_ptr(), stream))
        if world > 1:
            gather(st.y)

    def iters_executed(state):
        na = state.nactive.cpu().numpy()
        return int(np.sum(na[:nIter] > 0))

    for _ in range(max(3, warmup)):
        step_device()
    barrier()
    its = int(allmax(iters_executed(st)))       # job-level: the slowest shard decides when the loop is over
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    clk = ClockSampler(ctx.local) if headline else None
    if clk:
        clk.__enter__()
    barrier()
    t_wall0 = time.perf_counter()
    for s in range(steps):
        flush.fill_(s & 0xFF)           # L2 flush between timed iterations (untimed)
        ev[s][0].record()
        step_device()
        ev[s][1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    if clk:
        clk.__exit__()
    if dump_dir and rank == 0:      # before the passes below overwrite the state
        dump_outputs(dump_dir, st)
    ms_per_step = allmax(sum(a.elapsed_time(b) for a, b in ev)) / steps
    value = Bglob * its / (ms_per_step * 1e-3)

    # ---- the same loop replayed from a CUDA graph (icnn_loop_graph_*): device time and HOST enqueue time of both
    # forms -- what "launch-bound or not" means for this workload (VERDICT r01 item 5)
    loop_graph = None
    if world == 1 and os.environ.get("ICNN_BENCH_GRAPH", "1") != "0":
        gh = st.loop_graph(fg, ccfg)
        gsteps = steps if ms_per_step < 200.0 else min(steps, 3)

        def step_graph():
            st.y.copy_(y0_dev)
            _capi.check(_capi.lib.icnn_loop_graph_launch(gh, stream))

        def enqueue_ms(fn, reps=3):
            tt = 0.0
            for _ in range(reps):
                torch.cuda.synchronize()
                t0_ = time.perf_counter()
                fn()
                tt += time.perf_counter() - t0_
            torch.cuda.synchronize()
            return tt / reps * 1e3
        for _ in range(2):
            step_graph()
        torch.cuda.synchronize()
        gev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(gsteps)]
        for s in range(gsteps):
            flush.fill_(s & 0xFF)
            gev[s][0].record()
            step_graph()
            gev[s][1].record()
        torch.cuda.synchronize()
        loop_graph = {"ms_per_step": sum(a.elapsed_time(b) for a, b in gev) / gsteps, "eager_ms_per_step": ms_per_step,
                      "steps": gsteps, "kernel_nodes": int(_capi.lib.icnn_loop_graph_nodes(gh)),
                      "host_enqueue_ms": {"eager": enqueue_ms(step_device), "graph": enqueue_ms(step_graph)}}

    # ---- end to end through the public API, host buffers -------------------------------------
    def step_e2e():
        if world > 1 and strong:
            # the public multi-GPU entry: shards the HOST batch, binds, solves, all-gathers y*
            yall, out = idist.solve_batch_sharded(net, x_all_pin, y0_all_pin, nIter=nIter, solver=solver,
                                                  variant=variant, affine=cfg["affine"], state=st)
            return yall, st
        fg_h = net.bind(x_pin, affine=cfg["affine"])            # H2D x + x-path gate precompute
        out = bundle_entropy.solveBatch(fg_h, y0_work, nIter=nIter, solver=solver, variant=variant,
                                        return_state=True, state=st)   # H2D y0 ... D2H y* (into y0_work, pinned)
        if world > 1:
            gather(out[-1].y)
        return None, out[-1]

    if world > 1 and strong:
        x_all_pin = torch.from_numpy(np.ascontiguousarray(x_all, dtype=np.float32)).pin_memory()
        y0_all_pin = torch.from_numpy(np.ascontiguousarray(y0_all)).pin_memory()
    y0_work = torch.empty_like(y0_pin).pin_memory()
    for _ in range(2):
        y0_work.copy_(y0_pin)
        step_e2e()
    barrier()
    e2e_t = 0.0
    for s in range(steps):
        y0_work.copy_(y0_pin)           # solveBatch overwrites initXs in place like the reference; restore (untimed)
        barrier()
        t0 = time.perf_counter()
        _ya, st_e = step_e2e()
        torch.cuda.synchronize()
        e2e_t += time.perf_counter() - t0
    e2e_s = allmax(e2e_t / steps)
    its_e2e = int(allmax(iters_executed(st_e)))
    e2e = dict(value=Bglob * its_e2e / e2e_s, unit=UNIT, ms_per_step=e2e_s * 1e3,
               h2d_bytes_per_step=int(x_pin.numel() * 4 + y0_pin.numel() * 8),
               d2h_bytes_per_step=int(B * n * 8 + B * 4 * 2 + (nIter + 1) * 4),
               api=("icnn_b200.dist.solve_batch_sharded" if (world > 1 and strong)
                    else "icnn_b200.bundle_entropy.solveBatch(PICNN.bind(x_host), y0_host, state=reused)"))

    # ---- instrumented pass: per-kernel-class CUDA-event time (K1 = PICNN f/grad, K2 = bundle step) and the
    # per-iteration statistics the roofline's algorithmic work is computed from
    # pass 0: statistics on (atomics into iter_stats), its timings are kept only as a cross-check; passes 1..2: statistics off
    # (the timed path), K1 / K2 times averaged
    reps = 2
    k1_ms = k2_ms = 0.0
    k2_ms_stats = 0.0
    for rep in range(reps + 1):
        st.c.iter_stats = stats_ptr if rep == 0 else None
        st.y.copy_(y0_dev)
        _capi.check(_capi.lib.icnn_bundle_init(C.byref(st.c), nIter, stream))
        evs = []
        for t in range(its):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            _capi.check(_capi.lib.icnn_picnn_fg(net._h, C.byref(fg.c_gates), st.y32.data_ptr(), st.f.data_ptr(),
                                                st.G.data_ptr(), 0, st.perm.data_ptr(), st.count.data_ptr(), KS,
                                                fg.ws.data_ptr(), None, stream))
            e1.record()
            _capi.check(_capi.lib.icnn_bundle_step(C.byref(ccfg), C.byref(st.c), t, stream))
            e2.record()
            evs.append((e0, e1, e2))
        torch.cuda.synchronize()
        if rep == 0:
            k2_ms_stats = sum(b.elapsed_time(c) for _, b, c in evs)
        else:
            k1_ms += sum(a.elapsed_time(b) for a, b, _ in evs) / reps
            k2_ms += sum(b.elapsed_time(c) for _, b, c in evs) / reps
    stats = st.iter_stats.cpu().numpy()
    st.c.iter_stats = None
    ksum = int(st.ksum.sum().item())
    solves_local = int(stats[:, 0].sum())            # samples x iterations actually entered on this rank
    peaks = ctx.peaks
    L = len(cfg["hidden"])
    tc_on = B >= 64 and not os.environ.get("ICNN_K1", "tc").startswith("s")
    small = n <= 8 and KS <= 10
    k2_name = ("bundle_step_small_kernel (one thread per sample)" if small else
               "bundle_pc_kernel<8 warps, three n-vectors> (two-sweep PC, DMMA; two samples per SM)"
               if (solver == "pc" and variant == "lib" and 2048 < n <= 4096 and n % 4 == 0 and os.environ.get("ICNN_PC_V3", "") != "0")
               else "bundle_pc_kernel (two-sweep PC, DMMA)" if (solver == "pc" and variant == "lib" and (n <= 256 or n > 1024))
               else "bundle_step_kernel (DMMA Gram, FP64)")
    # K2: bound by the FP64 pipe (DMMA Gram + FP64 vector work); SURVEY.md 8d's HBM model kept beside it
    k2_flops = k2_fp64_flops(n, stats)
    k2_bytes = 4.0 * n * (ksum + 2.0 * B * its) + 8.0 * ksum
    tr = ctx.traffic.get(name, {})

    def _traffic(kname):
        t_ = tr.get(kname)
        if not t_:
            return None, None
        return t_["bytes"] * (float(B) / t_["rows"]), "%s; %d rows captured, scaled to %d rows (independent samples)" % (t_["source"], t_["rows"], B)
    roof_k2 = dict(kernel=k2_name, bound="tensor", pipe="fp64 tensor core (DMMA m8n8k4) + FP64 FMA",
                   achieved=k2_flops / (k2_ms * 1e-3) / 1e12, peak=ctx.fp64_peak, unit="TFLOP/s",
                   peak_source="measured live (icnn_fp64_mma_probe, DMMA)",
                   traffic=_traffic("K2")[0], traffic_source=_traffic("K2")[1],
                   launches=its, ms_per_launch=k2_ms / max(its, 1), share_of_step=k2_ms / (k1_ms + k2_ms),
                   ms_per_launch_with_statistics=k2_ms_stats / max(its, 1),
                   algorithmic_gflop_per_step=k2_flops / 1e9,
                   inner_iterations_per_solve=float(stats[:, 2].sum() / max(stats[:, 0].sum() - stats[:, 5].sum(), 1)),
                   mean_active_rows=float(stats[:, 1].sum() / max(stats[:, 0].sum() - stats[:, 5].sum(), 1)),
                   hbm_model=dict(bound="hbm", achieved=k2_bytes / (k2_ms * 1e-3) / 1e9, peak=peaks["hbm_gbs"],
                                  unit="GB/s", frac=k2_bytes / (k2_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                  note="SURVEY.md 8d single-pass bytes 4n(k_t+2)+8k_t per solve; the solve re-reads "
                                       "its rows from L2 2-5 times per interior-point iteration and is FP64-bound"))
    roof_k2["frac"] = roof_k2["achieved"] / roof_k2["peak"] if roof_k2["peak"] else None
    k1_flops = flop_fg(cfg) * B * its
    k1_name = ("tc_gemm_kernel (tcgen05 3xTF32 + TMA) + gate_y + out_layer" if tc_on
               else "gated_gemm_kernel + out_layer (FP32 FFMA)")
    nl_k1 = its * (2 * L + 2)
    roof_k1 = dict(kernel=k1_name, bound="tensor", achieved=k1_flops / (k1_ms * 1e-3) / 1e12,
                   peak=peaks["bf16_sustained"], unit="TFLOP/s", peak_source=peaks["source"] + ", bf16 sustained",
                   traffic=_traffic("K1")[0], traffic_source=_traffic("K1")[1],
                   launches=nl_k1, ms_per_launch=k1_ms / max(nl_k1, 1), share_of_step=k1_ms / (k1_ms + k2_ms),
                   note="FP32-accurate GEMMs as 3 TF32 MMAs per product: the ceiling of this formulation is "
                        "tf32 peak / 3 = bf16 peak / 6",
                   frac_of_3xtf32_ceiling=k1_flops / (k1_ms * 1e-3) / 1e12 / (peaks["bf16_sustained"] / 6.0))
    roof_k1["frac"] = roof_k1["achieved"] / roof_k1["peak"]
    dominant = dict(roof_k2 if k2_ms >= k1_ms else roof_k1)

    rec = {
        "workload": workload_string(name, cfg, solver), "value": value, "unit": UNIT, "ms_per_step": ms_per_step,
        "steps": steps, "iters_executed": its, "iters_requested": nIter, "global_batch": Bglob,
        "rows_per_gpu": B, "e2e": e2e, "roofline": dominant,
        "kernels": {"K1_picnn_fg": roof_k1, "K2_bundle_step": roof_k2},
        "gpu_launches_per_step": 2 + nIter * (2 * L + (3 if tc_on else 2)),
        "per_iteration": {"entering": stats[:its, 0].tolist(), "mean_k": (stats[:its, 1] / np.maximum(stats[:its, 0] - stats[:its, 5], 1)).round(2).tolist(),
                          "mean_f_minus_H": (stats[:its, 6] / np.maximum(stats[:its, 0], 1)).round(4).tolist()} if headline else None,
        "wall_s_timed_region": t_wall,
        "loop_graph": loop_graph,
    }
    if clk:
        rec["clocks"] = clk.summary()
    # what bounds strong scaling: K2 runs one CTA per sample, ceil(rows / resident CTAs) waves per launch -- with fewer rows
    # per GPU the last partial wave weighs more (wave quantisation); the all-gather of y* is one NCCL call per step
    try:
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        v3 = k2_name.startswith("bundle_pc_kernel<8 warps, three n-vectors>")
        if v3 and B > 0:
            resident = 2 * sms
            waves = -(-B // resident)
            rec["strong_scaling_model"] = {
                "limiting_kernel": "K2 " + k2_name, "resident_samples_per_gpu": resident, "rows_per_gpu": B,
                "waves_per_launch": waves, "wave_efficiency": B / float(resident * waves),
                "allgather_bytes_per_step": int(Bglob * n * 8) if world > 1 else 0}
    except Exception as exc:      # informational only
        rec["strong_scaling_model"] = {"error": repr(exc)}
    # ---- C3 (SURVEY.md 8d config 3 asks for both inner loops): 30-step momentum GD next to the bundle loop,
    # the final mean f(y) - H(y) of each (what ebundle-vs-gd.py:94-99 plots), and the GD training backward
    if name == "C3" and world == 1 and not cfg["affine"]:
        from icnn_b200 import gd as _gd, gd_grad as _gdg

        def f_minus_h(y32):
            f_, _g = fg.fg_device(y32.contiguous())
            ent = -(y32 * torch.log(y32) + (1 - y32) * torch.log(1 - y32))
            ent = torch.nan_to_num(ent, nan=0.0).sum(1)        # 0 log 0 = 0 (ebundle-vs-gd.py:38-41)
            return float((f_ - ent).mean())

        y0f = y0_dev.to(torch.float32)
        tYd = (torch.rand(B, n, device=dev, generator=torch.Generator(device=dev).manual_seed(5)) < 0.1).float()

        def timed(fn, reps=5):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0_.record()
            for _ in range(reps):
                r_ = fn()
            e1_.record()
            torch.cuda.synchronize()
            return e0_.elapsed_time(e1_) / reps, r_

        ms_gd, (y_gd, _f) = timed(lambda: _gd.solve(fg, y0f, nIter=30, lr=0.01, momentum=0.3, return_device=True))
        ms_bw, _r = timed(lambda: _gdg.gd_grad(fg, y0f, tYd, nIter=30, lr=0.01, momentum=0.3, return_device=True))
        step_device()
        torch.cuda.synchronize()
        rec["gd_mode"] = {"gd_inner_loop": {"iters": 30, "lr": 0.01, "momentum": 0.3, "ms": ms_gd,
                                            "value": B * 30 / (ms_gd * 1e-3), "unit": UNIT,
                                            "mean_f_minus_H": f_minus_h(y_gd),
                                            "roofline": {"bound": "tensor", "achieved": flop_fg(cfg) * B * 30 / (ms_gd * 1e-3) / 1e12,
                                                         "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                                                         "frac": flop_fg(cfg) * B * 30 / (ms_gd * 1e-3) / 1e12 / peaks["bf16_sustained"]}},
                          "bundle_inner_loop": {"iters": its, "mean_f_minus_H": f_minus_h(st.y.to(torch.float32))},
                          "gd_training_backward_ms": ms_bw}
    if rank == 0 and cpu_seconds > 0 and world == 1:
        rec["cpu_baseline"] = cpu_baseline(name, cpu_seconds, reference_cost=headline)
        rec["e2e_over_cpu"] = e2e["value"] / rec["cpu_baseline"]["value"]
    del st, fg, net
    torch.cuda.empty_cache()
    return rec


def run_gpu(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from icnn_b200 import workloads

    ctx = Ctx()
    ctx.rank = int(os.environ.get("RANK", "0"))
    ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.local = int(os.environ.get("LOCAL_RANK", "0"))
    if ctx.world != args.gpus and ctx.rank == 0 and ctx.world == 1 and args.gpus > 1:
        print("bench.py: --gpus %d needs torchrun (WORLD_SIZE=1 seen)" % args.gpus, file=sys.stderr)
        sys.exit(2)
    torch.cuda.set_device(ctx.local)
    ctx.dev = torch.device("cuda", ctx.local)
    if ctx.world > 1:
        dist.init_process_group("nccl", device_id=ctx.dev)
    ctx.flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=ctx.dev)   # > 126 MB L2
    ctx.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ctx.peaks = load_peaks()
    ctx.traffic = load_traffic()
    ctx.fp64_peak = measure_fp64_peak(ctx)
    scaling = args.scaling or "strong"
    cpu_s = 0.0 if args.no_cpu_baseline else args.cpu_seconds
    head = measure_workload(ctx, args.workload, args.steps, max(3, args.warmup), scaling, args.solver, cpu_s, True,
                            args.dump_outputs)
    subs = {}
    if ctx.world == 1 and not args.no_sub:
        for w in SUB_WORKLOADS:
            if w == args.workload:
                continue
            subs[w] = measure_workload(ctx, w, args.sub_steps, 3, "strong", args.solver,
                                       0.0 if args.no_cpu_baseline else args.sub_cpu_seconds, False)
    if ctx.world > 1:
        dist.barrier()
    line = None
    if ctx.rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32 (K1 PICNN f/grad) + f64 (K2 bundle solve)",
            "data": "synthetic", "impl": "icnn_b200",
            "config": {"workload": head["workload"], "global_batch": head["global_batch"],
                       "rows_per_gpu": head["rows_per_gpu"],
                       "iters_executed": head["iters_executed"], "iters_requested": head["iters_requested"],
                       "parallelism": ("sample-sharded x%d (%s scaling), one all-gather of y*" % (ctx.world, scaling)),
                       "l2": "512 MiB buffer written between timed steps (L2 flush)",
                       "wall_s_timed_region": head["wall_s_timed_region"]},
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches_per_step"] * args.steps,
            "clocks": head.get("clocks"), "roofline": head["roofline"], "kernels": head["kernels"],
            "cpu_baseline": head.get("cpu_baseline"), "e2e_over_cpu": head.get("e2e_over_cpu"),
            "per_iteration": head["per_iteration"], "loop_graph": head.get("loop_graph"),
            "strong_scaling_model": head.get("strong_scaling_model"),
            "fp64_mma_peak_tflops": ctx.fp64_peak,
            "configs": subs,
            "target_shape": subs.get("T"),
        }
        print(json.dumps(line))
    if ctx.world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def run_reference(args):
    """The reference's CPU path (oracle port, all host cores) on the same config/metric.  Loads no native code."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from icnn_b200 import workloads
    cfg = workloads.CONFIGS[args.workload]
    procs = usable_cores()
    total_steps = args.steps + args.warmup
    per_step_budget = max(1.5, min(20.0, 150.0 / max(total_steps, 1)))
    rows, its, _ = cpu_plan(args.workload, procs, per_step_budget)     # fixed sample for every step
    for _ in range(args.warmup):
        cpu_reference(args.workload, rows, procs, nIter=its)
    per_step = []
    solves = 0
    for _ in range(args.steps):
        s, w = cpu_reference(args.workload, rows, procs, nIter=its)
        solves = s
        per_step.append(w)
    med = float(np.median(per_step))
    value = solves / med
    sample = ("%d of %d rows x %d of %d iterations per step (median of %d steps; mean-based value %.1f), numpy oracle "
              "port of lib/bundle_entropy.solveBatch(solver='pc') / the RL copy for C4 with float32-arithmetic fg, "
              "%d processes x 1 BLAS thread" % (rows, cfg["B"], its, cfg["nIter"], args.steps,
                                                solves * len(per_step) / sum(per_step), min(procs, rows)))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True,
            "scaling": args.scaling or "strong", "vs_baseline": None, "dtype": "f64 solver / f32 fg",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_string(args.workload, cfg)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": min(procs, rows), "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "native_modules_loaded": sorted(m for m in sys.modules if m.startswith("icnn_b200._capi"))}
    print(json.dumps(line))


def main():
    # the benchmark writes nothing into the tree it runs from (which may be read-only): no __pycache__ beside the
    # sources, here or in the CPU arm's worker processes (they inherit the environment)
    sys.dont_write_bytecode = True
    os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="icnn_b200", choices=["icnn_b200", "reference"])
    ap.add_argument("--workload", default="C5", choices=["C1", "C2", "C3", "C4", "C5", "T"])
    ap.add_argument("--solver", default="pc", choices=["pc", "newton"])
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="strong (default): the workload's batch sharded over the GPUs; weak: the batch per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-records of the other configs")
    ap.add_argument("--no-target-shape", action="store_true", help="alias of --no-sub (round-1 flag)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--sub-cpu-seconds", type=float, default=6.0)
    ap.add_argument("--sub-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline workload's outputs of the last timed step (rank 0's rows) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.sub_steps < 1:
        ap.error("--steps and --sub-steps must be >= 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none to write")
    args.no_sub = args.no_sub or args.no_target_shape
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_gpu(args)
    finally:
        _close_pools()


if __name__ == "__main__":
    main()
