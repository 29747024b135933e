#!/usr/bin/env python
"""Benchmark of the ideal-ballooning hot path: field-line solves/sec (fp64, lambda_max + eigenvector).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload d3d|ncsx|hberg|salpha|adjoint] [--equilibria E] [--strong] [--dump-outputs DIR]

One *step* = one pass of the hot path over one batch of synthetic input; ``--steps`` is the number of timed steps.  The
inputs are seeded: the same arguments give the same inputs in every run, and ``--dump-outputs`` stores what the last timed
step computed, so that two builds can be compared output for output.

scan workloads (BASELINE.json configs[1..3]; default ``d3d`` = configs[1], the config the metric is quoted on):
    K1 geometry (ns x nalpha field lines) -> K2+K3 with the guarded per-surface arg-max fused into the solver kernel
    (ns x nalpha x nth0 solves, lambda + eigenvector of every solve) -> (N > 1: ONE all_gather_into_tensor of the packed
    per-surface (max, index) pairs, written by the kernel straight into the send slot).
    ``--equilibria E`` independently perturbed equilibria are batched per step (the reference scans totalndofs+1 perturbed
    equilibria per outer iteration, sims_runner_D3D.py:109); the default line also carries ``single_equilibrium`` = the
    config exactly as BASELINE states it (E = 1).  Weak scaling: every rank scans its own equilibria.  ``--strong``: ONE
    batch of surfaces sharded over the ranks in contiguous blocks (scan.shard_range), total work fixed.
``salpha`` (configs[0]): the 200 x 100 x 3 (shat, alpha, theta0) grid of bishop_ball_s-alpha.py:213-229 through K2+K3 from
    explicit g, c, f; unstable <=> lambda_max > 0, OR over theta0 (:282-289).
``adjoint`` (configs[4]): lambda_max + eigenvector + (dlam/dalpha, dlam/dtheta0) for NCSX-like field lines with i.i.d.
    (s, alpha, theta0): K1 for the three lines alpha -+ del/2 of every point -> K2+K3 on the centre line -> K4
    (obj_w_grad contraction) -> (N > 1: all-gather of the gradients, 16 B per point).  131 072 points per GPU = the
    per-GPU share of the 1 M-line batch on 8 GPUs.

``value``    device-timed throughput (CUDA events on the launching stream), inputs resident in HBM, L2 flushed between steps.
``e2e``      the same metric through the public host-buffer API (pinned host buffers in, results out, copies inside the
             timing): scan workloads = the C-ABI call ``ibs_scan_host``.
``roofline`` the solver kernel (K2+K3): algorithmic bytes 32*N per solve / its CUDA-event time vs the measured HBM copy
             bandwidth of MEASURED_PEAKS.json.  ``roofline_fp64``: the same kernel (and K1) against the FP64 FMA peak
             measured live by the library's DFMA probe -- the pipe these kernels are actually bound by.
``cpu_baseline`` / ``--impl reference``: the reference's own numpy/scipy functions (unmodified utils.py from oracle/_ref,
             kind "reference"; the oracle port if that copy is absent, kind "port") on the host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "field-line ballooning solves/sec (fp64, lambda_max+eigvec)"
WORKLOADS = {
    #          kind    ns   nalpha nth0 ntheta span(pi)
    "d3d":   ("d3d",   128, 1,     64,  1024,  4),
    "ncsx":  ("ncsx",  64,  32,    32,  2048,  4),
    "hberg": ("hberg", 256, 64,    1,   8192,  8),
}
SALPHA = dict(nshat=200, nalpha=100, theta0=(0.0, 0.1, 0.2), ntheta=1024, span=10)     # bishop_ball_s-alpha.py:213-229
ADJOINT = dict(kind="ncsx", ntheta=1024, span=4, points=131072, del_alpha=0.004)        # utils.py:1639
ALL_WORKLOADS = sorted(WORKLOADS) + ["salpha", "adjoint"]


def scan_eligible(nth0, N):
    """Mirrors scan_solver_eligible (ibs_scan_solver.cu): which K2+K3 kernel a scan-shaped batch is dispatched to."""
    return os.environ.get("IBS_SCAN", "1") != "0" and nth0 >= 4 and (N & 1) == 1 and N >= 65


def scan2_size_ok(N):
    """Mirrors scan2_size_ok (ibs_scan2_core.cuh): the lane-per-chain kernel needs N - 1 (and the coarsest level's) to be a multiple of 16."""
    nlev = 0
    while nlev < 4 and (N - 1) % (2 << nlev) == 0 and ((N - 1) >> (nlev + 1)) + 1 >= 65:
        nlev += 1
    return N % 2 == 1 and N >= 65 and (N - 1) % 16 == 0 and ((N - 1) >> nlev) % 16 == 0 and os.environ.get("IBS_SCAN2", "1") != "0"


def solver_kernel_name(nth0, N):
    if not scan_eligible(nth0, N):
        return "solve_kernel (K2+K3, team per solve)"
    return "scan2_solve_kernel (K2+K3, lane per chain)" if scan2_size_ok(N) else "scan_solve_kernel (K2+K3, lane per solve)"


def workload_grids(name):
    if name == "salpha":
        theta = np.linspace(-SALPHA["span"] * np.pi, SALPHA["span"] * np.pi, SALPHA["ntheta"] + 1)
        return "salpha", np.linspace(0.0, 2.0, SALPHA["nshat"]), np.linspace(0.0, 1.2, SALPHA["nalpha"]), np.array(SALPHA["theta0"]), theta
    if name == "adjoint":
        theta = np.linspace(-ADJOINT["span"] * np.pi, ADJOINT["span"] * np.pi, ADJOINT["ntheta"] + 1)
        return ADJOINT["kind"], np.array([0.5, 0.95]), np.array([0.0, np.pi]), np.array([0.0, 0.5 * np.pi]), theta
    kind, ns, na, nt, nth, span = WORKLOADS[name]
    s = np.linspace(0.5, 0.95, ns)                                   # ball_scan.py:197
    alpha = np.linspace(0.0, np.pi, na) if na > 1 else np.array([0.0])
    theta0 = np.linspace(0.0, 0.5 * np.pi, nt) if nt > 1 else np.array([0.0])
    theta = np.linspace(-span * np.pi, span * np.pi, nth + 1)        # ntheta intervals -> N = ntheta+1 points
    return kind, s, alpha, theta0, theta


def build_tables(name, equilibria, seed0):
    """Host-side setup (not timed): synthetic equilibria -> radial splines -> per-surface tables."""
    import dataclasses
    from ideal_ballooning_solver_b200 import synthetic, tables
    kind, s, alpha, theta0, theta = workload_grids(name)
    parts = [tables.RadialSplines(synthetic.make_equilibrium(kind, seed=seed0 + e)).evaluate(s) for e in range(equilibria)]
    st = dataclasses.replace(parts[0], tab_mn=np.concatenate([p.tab_mn for p in parts]),
                             tab_nyq=np.concatenate([p.tab_nyq for p in parts]),
                             scal=np.concatenate([p.scal for p in parts]),
                             bsupumnc=None if parts[0].bsupumnc is None else np.concatenate([p.bsupumnc for p in parts]))
    return st, alpha, theta0, theta


def describe(workload, equilibria=1, points=None, strong=False):
    if workload == "salpha":
        return (f"s-alpha shifted-circle model (tests/shifted-circle-s-alpha): {SALPHA['nshat']} shat x {SALPHA['nalpha']} alpha x "
                f"{len(SALPHA['theta0'])} theta0, ntheta={SALPHA['ntheta']} (N={SALPHA['ntheta'] + 1} points, theta in +-{SALPHA['span']}pi)")
    if workload == "adjoint":
        return (f"adjoint gradient batch: lambda_max + eigvec + (dlam/dalpha, dlam/dtheta0) for {points} NCSX-like field lines per GPU, "
                f"(s, alpha, theta0) i.i.d. uniform, ntheta={ADJOINT['ntheta']} (N={ADJOINT['ntheta'] + 1} points); 131072 = the per-GPU "
                f"share of the 1M-line batch on 8 GPUs")
    kind, ns, na, nt, nth, span = WORKLOADS[workload]
    how = "ONE batch sharded over the ranks by surface blocks" if strong else "per step per GPU"
    return (f"{kind.upper()}-like synthetic VMEC-shaped scan: {ns} surfaces x {na} alpha x {nt} theta0, ntheta={nth} "
            f"(N={nth + 1} points, theta in +-{span}pi), x {equilibria} equilibria {how}")


_JSON_FD = None


def claim_stdout():
    """Everything a library prints on fd 1 (NCCL's version banner under NCCL_DEBUG=VERSION/WARN, ...) goes to stderr from here
    on; ``emit`` writes the ONE JSON line on the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def traffic_per_solve(workload):
    """ncu dram bytes per solve of the dominant solver kernel (profiles/roofline_traffic.json), or None."""
    rf = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        return float(json.load(open(rf))[workload]["dram_bytes_per_solve"])
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        if os.environ.get("IBS_BENCH_NO_SAMPLER"):       # diagnostic: is a slow step caused by the nvidia-smi queries?
            return
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        # nvidia-smi's start-up (driver handshake, first query) stalls the device for tens of ms: let it finish BEFORE the
        # warm-up starts, i.e. wait for its first sample (its steady-state queries do not perturb the steps: checked with
        # IBS_BENCH_NO_SAMPLER=1)
        t0 = time.perf_counter()
        while self.p is not None and self.p.poll() is None and time.perf_counter() - t0 < 3.0:
            try:
                if os.path.getsize(self.f.name) > 0:
                    break
            except OSError:
                break
            time.sleep(0.02)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's own numpy/scipy path on the host cores (the unmodified utils.py from oracle/_ref when the
# recipe oracle/make_ref.py has been run -- kind "reference" -- else the oracle port of the same algorithm -- kind "port")
# ---------------------------------------------------------------------------------------------------
_W = {}          # per-worker state (filled by _cpu_init in every pool process)


def _one_thread():
    os.environ["OMP_NUM_THREADS"] = os.environ["OPENBLAS_NUM_THREADS"] = "1"     # slurm_ball_scan_template.sl:10
    try:
        from threadpoolctl import threadpool_limits
        _W["limit"] = threadpool_limits(1)
    except Exception:
        pass


def _cpu_init(workload, kind_cpu):
    """Pool initialiser: imports and the per-equilibrium set-up (radial splines), none of it timed."""
    _one_thread()
    import warnings
    warnings.simplefilter("ignore")
    from ideal_ballooning_solver_b200 import synthetic, tables
    kind, s, alpha, theta0, theta = workload_grids(workload)
    _W.update(kind_cpu=kind_cpu, s=s, theta=theta, workload=workload)
    if kind_cpu == "reference":
        from oracle import ref_shim
        _W["u"] = ref_shim.load_reference_utils()
    else:
        from oracle import ballooning_oracle as bo
        _W["bo"] = bo
    if workload == "salpha":
        return
    wout = synthetic.make_equilibrium(kind, seed=12345)
    if kind_cpu == "reference":
        from oracle import ref_shim
        _W["vs"] = _W["u"].vmec_splines(ref_shim.FakeVmec(wout))                 # utils.py:37 (once per equilibrium)
    else:
        _W["splines"] = tables.RadialSplines(wout)
        _W["st"] = _W["splines"].evaluate(s) if workload != "adjoint" else None


def _cpu_warm(_):
    time.sleep(0.05)          # let every worker take one of these, so that all of them are initialised before the clock starts
    return os.getpid()


def _vguess(theta):
    return (1 - np.tanh(theta[1:-1] / np.pi) ** 2) * np.cos(theta[1:-1] / (2 * max(1, int(round(theta[-1] / np.pi)))))      # ball_scan.py:209


def _cpu_task(args):
    """scan workloads: one field line = geometry (vmec_fieldlines) + the theta0 loop of gamma_ball_full calls with the start
    vector chained (ball_scan.py:251-274).  salpha: gamma_ball_full on the analytic coefficients.  adjoint: obj_w_grad
    (three field lines + one solve + the adjoint integrals, utils.py:1632-1728).  By the reference's own functions or by
    their oracle port."""
    theta = _W["theta"]
    vg = _vguess(theta)
    ref = _W["kind_cpu"] == "reference"
    t0 = time.perf_counter()
    n = 0
    if _W["workload"] == "salpha":
        shat, alpha, theta0s = args
        for th0 in theta0s:
            lam_ = shat * (theta - th0) - alpha * (np.sin(theta) - np.sin(th0))
            g = 1.0 + lam_ * lam_
            cv = np.cos(theta) + np.sin(theta) * lam_
            one = np.ones_like(theta)
            a = (-alpha, theta, one, one, cv, g, vg, 2.0)
            lam, X, *_ = _W["u"].gamma_ball_full(*a) if ref else _W["bo"].gamma_ball_full(*a, tol=5.0e-7, method="arpack")
            n += 1
    elif _W["workload"] == "adjoint":
        s_val, alpha, th0 = args
        if ref:
            _W["u"].obj_w_grad((alpha, th0), _W["vs"], s_val, theta, vg, 1.0)
        else:
            bo = _W["bo"]
            st1 = _W["splines"].evaluate(np.array([s_val]))
            bo.obj_w_grad((alpha, th0), lambda a: bo.fieldlines(st1, np.atleast_1d(a), theta), theta, vg, 1.0)
        n = 1
    elif ref:
        js, alpha, theta0s = args
        u = _W["u"]
        fl = u.vmec_fieldlines(_W["vs"], float(_W["s"][js]), float(alpha), theta1d=theta)
        bmag, gradpar = fl.bmag[0][0], fl.gradpar_theta_pest[0][0]
        dP = -0.5 * np.mean((fl.cvdrift[0][0] - fl.gbdrift[0][0]) * bmag ** 2)                  # ball_scan.py:262
        for th0 in theta0s:
            cv = fl.cvdrift[0][0] + th0 * fl.cvdrift0[0][0]                                       # ball_scan.py:267-268
            gd = fl.gds2[0][0] + 2 * th0 * fl.gds21[0][0] + th0 ** 2 * fl.gds22[0][0]
            lam, X, *_ = u.gamma_ball_full(dP, theta, bmag, gradpar, cv, gd, vg, 1.0)           # ball_scan.py:269
            vg = X[1:-1]
            n += 1
    else:
        js, alpha, theta0s = args
        bo = _W["bo"]
        fl = bo.fieldlines(_W["st"].select([js]), np.array([alpha]), theta)
        dP = bo.dpdrho_of(fl)
        for th0 in theta0s:
            cv, gd = bo.theta0_shift(fl, th0)
            lam, X, *_ = bo.gamma_ball_full(dP, theta, fl.bmag[0][0], fl.gradpar_theta_pest[0][0], cv, gd, vg, 1.0,
                                            tol=5.0e-7, method="arpack")
            vg = X[1:-1]
            n += 1
    return n, time.perf_counter() - t0


def cpu_kind():
    from oracle import ref_shim
    return "reference" if ref_shim.reference_available() else "port"


def cpu_reference_rate(workload, lines_per_core=None, solves_per_line=6, cores=None):
    """Solves/s of the reference algorithm on the host cores for a bounded sample of `workload`.  The pool's start-up
    (process creation, imports, spline set-up) is outside the timed region; every core gets `lines_per_core` tasks."""
    import multiprocessing as mp
    kind_cpu = cpu_kind()
    kind, s, alpha, theta0, theta = workload_grids(workload)
    N = len(theta)
    cores = cores or os.cpu_count() or 1
    if N > 4200:
        # dense (N-2)^2 matrix = 0.5 GB and an O(N^3) LU per solve (utils.py:1584-1597): a handful of solves only
        cores = max(1, min(cores, 4))
        lines_per_core, solves_per_line = 1, 1
    elif lines_per_core is None:
        lines_per_core = 4 if N <= 1100 else 2
    ntask = cores * lines_per_core
    rng = np.random.default_rng(0)
    if workload == "salpha":
        pick = theta0
        tasks = [(float(rng.choice(s)), float(rng.choice(alpha)), pick) for _ in range(ntask * 2)]
        unit = f"{len(tasks)} (shat, alpha) points x {len(pick)} theta0"
    elif workload == "adjoint":
        tasks = [(float(rng.uniform(0.5, 0.95)), float(rng.uniform(0, np.pi)), float(rng.uniform(0, 0.5 * np.pi))) for _ in range(ntask)]
        unit = f"{len(tasks)} obj_w_grad points (3 field lines + 1 solve + adjoint integrals each)"
    else:
        pick = np.asarray(theta0[np.linspace(0, len(theta0) - 1, min(solves_per_line, len(theta0))).astype(int)])
        tasks = [(int(rng.integers(0, len(s))), float(alpha[k % len(alpha)]), pick) for k in range(ntask)]
        unit = f"{len(tasks)} field lines x {len(pick)} theta0"
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init, initargs=(workload, kind_cpu)) as pool:
        pool.map(_cpu_warm, range(4 * cores), chunksize=1)
        t0 = time.perf_counter()
        res = pool.map(_cpu_task, tasks, chunksize=1)
        wall = time.perf_counter() - t0
    nsolve = sum(r[0] for r in res)
    percore = nsolve / sum(r[1] for r in res)
    what = ("the UNMODIFIED reference (oracle/_ref/utils.py: vmec_fieldlines + gamma_ball_full / obj_w_grad" if kind_cpu == "reference"
            else "oracle port of the reference algorithm (numpy geometry + dense matrix + ARPACK shift-invert")
    sample = (f"{unit} of the {workload} workload (N={N} points): {what}, tol=5e-7), "
              f"{cores} processes x 1 BLAS thread, pool start-up and spline set-up not timed; {percore:.2f} solves/s/core")
    return nsolve / wall, cores, sample, wall, kind_cpu


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    t_all = time.perf_counter()
    steps = args.steps
    for _ in range(steps):
        v, cores, sample, wall, kind_cpu = cpu_reference_rate(args.workload)
        vals.append(v)
    value = float(np.median(vals))
    line = {"metric": METRIC, "value": value, "unit": "solves/s",
            "impl": "reference", "n_gpus": args.gpus, "steps": steps, "warmup": 0,
            "ms_per_step": 1e3 * (time.perf_counter() - t_all) / steps, "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": describe(args.workload, args.equilibria, args.points, args.strong)},
            "cpu_baseline": {"value": value, "unit": "solves/s", "cores": cores, "kind": kind_cpu, "sample": sample},
            "e2e": {"value": value, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
class Harness:
    """Process-group set-up, the timed loop (CUDA events per stage, L2 flush between steps, max over ranks), clocks."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from ideal_ballooning_solver_b200 import _lib
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the one JSON line
            torch.cuda.set_device(local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        self.dev = torch.device("cuda", local_rank if self.world > 1 else torch.cuda.current_device())
        torch.cuda.set_device(self.dev)
        _lib.load(build_if_missing=True)
        self.flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=self.dev)     # > 126 MB L2
        self.sampler = None
        self.is_last = False
        self.last_out = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def timed(self, step, nstage, steps=None, warmup=None, sample_clocks=True, keep_last=False):
        """`step(timers)` records nstage+1 events.  Returns (total seconds = max over ranks of the summed step times, per-stage
        ms array (steps, nstage), per-step ms, wall seconds).  `keep_last`: what the last timed step returned is left in
        ``self.last_out`` (for --dump-outputs; the caller clears it)."""
        torch = self.torch
        steps = steps or self.args.steps
        warmup = max(self.args.warmup, 3) if warmup is None else warmup
        # the clock sampler starts BEFORE the warm-up (nvidia-smi's start-up stalls the device for a few ms)
        if sample_clocks and self.rank == 0 and self.sampler is None:
            self.sampler = ClockSampler(torch.cuda.current_device())
        # Everything that is not a step happens BEFORE the warm-up -- event creation, a generational collection of the
        # interpreter (10-100 ms when it strikes inside a step) -- so that the warm-up runs straight into the timed steps: an
        # idle gap of tens of ms between them made the first timed step take 4-80 ms instead of 3.6.  (The first step after the
        # barrier still runs 5-30 % slow -- IBS_BENCH_DUMP_STEPS=1 prints the slowest steps and their stages; more warm-up steps,
        # events recorded in the warm-up, synchronisations or idle gaps later in the loop do not reproduce it.)
        ev = lambda: torch.cuda.Event(enable_timing=True)
        timers = [[ev() for _ in range(nstage + 1)] for _ in range(steps)]
        import gc
        gc.collect()
        gc_was = gc.isenabled()
        gc.disable()
        try:
            # Power-state ramp, before the W warm-up steps: the process has just spent seconds on the host (tables), the device
            # sits in a low-power state, and the switch back (memory clocks included) takes longer than 3 steps -- it then
            # stalled the FIRST timed step for 5-140 ms in one run out of three.  Untimed steps until 0.3 s have gone by.
            t_ramp = time.perf_counter()
            for _ in range(400):
                step(None)
                self.flush.zero_()
                if _ % 8 == 7:
                    torch.cuda.synchronize()
                    # (every rank must run the same number of steps -- a step may hold a collective: the ranks agree on "time is up")
                    if self.max_over_ranks(time.perf_counter() - t_ramp) > float(os.environ.get("IBS_BENCH_RAMP_S", "0.3")):
                        break
            for _ in range(warmup):
                step(None)
                self.flush.zero_()
            self.barrier()
            t_wall = time.perf_counter()
            for k in range(steps):
                self.is_last = k == steps - 1
                out = step(timers[k])
                if not self.is_last:
                    out = None                  # released right away, so every step reuses the blocks the previous one freed
                self.flush.zero_()              # L2 flush between timed iterations (outside the event brackets)
            self.is_last = False
            self.last_out = out if keep_last else None
            self.barrier()
        finally:
            if gc_was:
                gc.enable()
        wall = time.perf_counter() - t_wall
        stage = np.array([[t[i].elapsed_time(t[i + 1]) for i in range(nstage)] for t in timers])
        total = np.array([t[0].elapsed_time(t[nstage]) for t in timers])
        if os.environ.get("IBS_BENCH_DUMP_STEPS"):       # diagnostic: which steps are the slow ones, and in which stage
            big = np.argsort(total)[-3:][::-1]
            print("slowest steps:", [(int(k), round(float(total[k]), 3), [round(float(x), 3) for x in stage[k]]) for k in big], file=sys.stderr)
        return self.max_over_ranks(total.sum()) * 1e-3, stage, total, wall

    def clocks(self):
        c = self.sampler.stop() if self.sampler else None
        self.sampler = None
        return c

    def finish(self, line):
        if self.rank == 0 and line is not None:
            emit(line)
        if self.world > 1:
            self.dist.destroy_process_group()


def rec(t, ev_idx):
    if t is not None:
        t[ev_idx].record()


def dump_outputs(dirname, arrays, limit=60 << 20):
    """``--dump-outputs``: write each device tensor of ``arrays`` (one row per solve / point / surface on axis 0) as
    ``dirname/<name>.npy`` in float64, under ``limit`` bytes in all.  Smallest first, an array is stored whole when it fits
    an equal share of what is left, else as the rows of a fixed seeded sample (their indices in ``<name>_rows.npy``): the
    same arguments always store the same elements, so two builds can be compared output for output."""
    import torch
    os.makedirs(dirname, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = limit
    for i, (name, t) in enumerate(items):
        share = left // (len(items) - i)
        if 8 * t.numel() > share:
            row = 8 * t[0].numel() + 8
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], share // row, replace=False))
            np.save(os.path.join(dirname, name + "_rows.npy"), rows.astype(np.float64))
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
            left -= 8 * len(rows)
        np.save(os.path.join(dirname, name + ".npy"), t.double().cpu().numpy())
        left -= 8 * t.numel()


def fp64_rooflines(H, entries):
    """entries: list of (kernel name, algorithmic FMAs per launch, ms per launch, note).  Peak measured live (DFMA probe)."""
    from ideal_ballooning_solver_b200 import engine
    peak = engine.fp64_peak_tflops(H.dev)
    out = []
    for name, fmas, ms, note in entries:
        ach = 2.0 * fmas / (ms * 1e-3) / 1e12
        out.append({"bound": "fp64", "kernel": name, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    "peak_source": "measured live: ibs_fp64_probe (independent DFMA chains, 32 warps/SM), CUDA events, best of 5",
                    "algorithmic_fma_per_launch": fmas, "kernel_ms": ms, "note": note})
    return out


def run_scan(H, args):
    torch = H.torch
    from ideal_ballooning_solver_b200 import engine, scan
    world, rank, dev = H.world, H.rank, H.dev
    kind, ns1, na, nt, nth, span = WORKLOADS[args.workload]
    N = nth + 1
    E = args.equilibria
    chain = scan.chain_length(nt if nt > 1 else na) if args.chain < 0 else max(1, args.chain)

    def make_case(E_, seed0, shard):
        st, alpha, theta0, theta = build_tables(args.workload, E_, seed0=seed0)
        ns_all = st.ns
        if shard:                                            # strong scaling: this rank's contiguous block of surfaces
            lo, hi = scan.shard_range(st.ns, rank, world)
            st = st.select(np.arange(lo, hi))
        ns = st.ns
        case = dict(st=st, ns=ns, ns_total=ns_all if shard else ns * world, alpha=alpha, theta0=theta0, theta=theta,
                    h=engine.grid_spacing(theta), dt=engine.DeviceTables.from_host(st, dev),
                    alpha_d=torch.from_numpy(alpha).to(dev), theta_d=torch.from_numpy(theta).to(dev),
                    th0_d=torch.from_numpy(theta0).to(dev).repeat(ns * na), nsolve=ns * na * nt, nlines=ns * na)
        # two exchange buffers used alternately: the all-gather of step k overlaps the kernels of step k + 1 (N > 1)
        case["gathers"] = [scan.SurfaceGather(case["ns_total"], dev) for _ in range(2 if world > 1 else 1)]
        case["gather"] = case["gathers"][0]
        case["nstep"] = 0
        return case

    def make_step(case):
        def step(t):
            gs = case["gathers"]
            g, g_prev = gs[case["nstep"] % len(gs)], gs[(case["nstep"] + 1) % len(gs)]
            case["nstep"] += 1
            rec(t, 0)
            geo = engine.geometry_batch(case["dt"], case["alpha_d"], case["theta_d"])
            rec(t, 1)
            g.wait()                             # (its exchange of two steps ago: long done)
            sol, best, sig = engine.scan_solve_argmax(geo.base, geo.dPdrho, case["th0_d"], case["h"], nt, na, want_X=True,
                                                      chain_len=chain, best_out=g.send)
            rec(t, 2)
            # N > 1: one all_gather_into_tensor of the packed (max, index) pairs, enqueued behind the solver and left to overlap
            # the next step's kernels; every step waits for the PREVIOUS step's exchange, the last timed step for its own too,
            # so all K exchanges complete inside the K timed brackets
            g.exchange(async_op=len(gs) > 1)
            if len(gs) > 1:
                g_prev.wait()
                if H.is_last:
                    g.wait()
            rec(t, 3)
            return sol, g.recv, sig
        return step

    main_case = make_case(E, 0 if args.strong else 1000 * rank, args.strong)
    step = make_step(main_case)
    sol = step(None)[0]
    torch.cuda.synchronize()
    nbad = int(np.count_nonzero((sol.info >> 16).cpu().numpy() & 3))
    mean_iters = float((sol.info & 0xFFFF).double().mean().item())
    total_s, stage, t_step, wall = H.timed(step, 3, keep_last=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        sol_l, surface_max, sig_l = H.last_out
        dump_outputs(args.dump_outputs, {"gamma": sol_l.lam, "X": sol_l.X, "flags": sol_l.info >> 16,
                                         "surface_max": surface_max.reshape(-1, 2), "sigma0": sig_l})
    H.last_out = sol_l = None
    nsolve_all = main_case["ns_total"] * na * nt
    value = nsolve_all * args.steps / total_s
    t_geo, t_solve, t_coll = stage[:, 0], stage[:, 1], stage[:, 2]

    # ---- the config exactly as BASELINE.json states it: ONE equilibrium per step
    single = None
    if not args.strong and E != 1 and not args.no_single:
        c1 = make_case(1, 777 + 1000 * rank, False)
        k1 = max(10, min(args.steps, 50))      # the secondary figures (this one, e2e) keep their own step counts
        tot1, st1, ts1, _ = H.timed(make_step(c1), 3, steps=k1, sample_clocks=False)
        single = {"value": c1["nsolve"] * world * k1 / tot1, "unit": "solves/s", "ms_per_step": 1e3 * tot1 / k1,
                  "solves_per_step_per_gpu": c1["nsolve"],
                  "kernel_ms": {"geometry": float(st1[:, 0].mean()), "solve": float(st1[:, 1].mean())},
                  "note": "one equilibrium = the BASELINE config as stated: %d (line, theta0-group) items for %d resident warps, so most "
                          "of the device idles; the reference itself scans ndofs+1 equilibria per outer iteration" %
                          (c1["nlines"] * ((nt + 31) // 32), 8 * torch.cuda.get_device_properties(dev).multi_processor_count)}
    clocks = H.clocks()

    # ---- end to end through the host-buffer C-ABI call (pinned host buffers, copies inside the timing)
    e2e = e2e_full = None
    st, alpha, theta0, theta = main_case["st"], main_case["alpha"], main_case["theta0"], main_case["theta"]
    ns, nsolve = main_case["ns"], main_case["nsolve"]
    if not args.no_e2e:
        import dataclasses
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
        st_p = dataclasses.replace(st, tab_mn=pin(st.tab_mn), tab_nyq=pin(st.tab_nyq), scal=pin(st.scal))
        out = dict(gamma=pin(np.empty((ns, na, nt))), val=pin(np.empty(ns)), sigma0=pin(np.empty(ns)),
                   idx=pin(np.empty(ns, dtype=np.int32)), xbest=pin(np.empty((ns, N))))
        a_p, t0_p, th_p = pin(alpha), pin(theta0), pin(theta)

        def e2e_run(reps, **kw):
            for _ in range(2):
                r = engine.scan_host(st_p, a_p, t0_p, th_p, out=out, **kw)
            H.barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                r = engine.scan_host(st_p, a_p, t0_p, th_p, out=out, **kw)
            return H.max_over_ranks(time.perf_counter() - t0), r

        h2d = st.tab_mn.nbytes + st.tab_nyq.nbytes + st.scal.nbytes + alpha.nbytes + theta.nbytes + theta0.nbytes
        ke = max(3, min(args.steps, 10))
        dt_e, r = e2e_run(ke, want_xbest=True)
        e2e = {"value": nsolve_all * ke / dt_e, "unit": "solves/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(8 * nsolve + ns * (8 + 8 + 4) + 8 * ns * N + 4),
               "eigvec": "arg-max only: the eigenfunction of each surface's maximum is returned (what ball_scan.py:322-339 keeps); "
                         "lambda of every solve is returned", "bad_solves": int(r[4]), "api": "ibs_scan_host (C ABI, host buffers)"}
        if not args.no_e2e_full and nsolve * N * 8 <= 6 << 30:
            out["xall"] = pin(np.empty((ns, na, nt, N)))
            kf = 3
            dt_f, r = e2e_run(kf, want_xbest=True, want_xall=True)
            e2e_full = {"value": nsolve_all * kf / dt_f, "unit": "solves/s", "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(8 * nsolve + ns * (8 + 8 + 4) + 8 * ns * N + 4 + 8 * nsolve * N),
                        "eigvec": "X of EVERY solve copied to the host (8 N bytes per solve over PCIe)"}
    if rank != 0:
        return H.finish(None)

    peak, peak_src = load_peaks()
    alg_bytes = 32.0 * N * main_case["nsolve"]                       # SURVEY 8(d): g, c, f in + X out per solve
    solve_ms = float(t_solve.mean())
    achieved = alg_bytes / (solve_ms * 1e-3) / 1e9
    tps = traffic_per_solve(args.workload)
    kname = solver_kernel_name(nt, N)
    # algorithmic FP64 work (DESIGN.md section 3): lane-per-solve kernel = 13 FMA per row and evaluation + 23 (Simpson pass)
    # + 15 (eigenfunction pass); team kernel ~ 22 per row and evaluation + 40; K1 = 10 mnmax + 9 mnmax_nyq FMAs per point
    rows = N * main_case["nsolve"]
    fma_solver = rows * ((13.0 * mean_iters + 38.0) if scan_eligible(nt, N) else (22.0 * mean_iters + 40.0))
    fma_geo = (10.0 * len(st.xm) + 9.0 * len(st.xm_nyq)) * N * main_case["nlines"]
    rf64 = fp64_rooflines(H, [(kname, fma_solver, solve_ms, "FMAs per solve = N x (13 x evaluations + 38) [lane kernel] or N x (22 x evaluations + 40) [team kernel]; kernel_ms includes the coefficient prep"),
                              ("geometry_kernel (K1)", fma_geo, float(t_geo.mean()), "algorithmic FMAs per point = 10 mnmax + 9 mnmax_nyq (SURVEY 8d); Newton and pointwise algebra not counted" +
                               ("; axisymmetric tables on a 2 pi-periodic theta grid: points one poloidal turn apart share their mode sums "
                                "(periodicity fold), so the EXECUTED mode-sum FMAs are ~1/%d of this algorithmic count" % max(1, int(round(span)))
                                if kind == "d3d" else ""))])
    launches = 6      # pack_mn, pack_nyq, geometry, dpdrho + (scan_prep, scan_solve [arg-max fused] | solve, argmax)
    line = {
        "metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": float(1e3 * total_s / args.steps), "higher_is_better": True, "scaling": "strong" if args.strong else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": describe(args.workload, E, strong=args.strong), "solves_per_step_per_gpu": main_case["nsolve"],
                   "field_lines_per_step_per_gpu": main_case["nlines"], "l2": "flushed between timed steps (256 MB write)",
                   "eigvec": "X written to HBM for every solve",
                   "mean_solver_iterations": mean_iters,      # fine-grid-equivalent evaluations per solve (output passes not counted)
                   "solver": kname, "argmax": "fused into the solver kernel's epilogue" if scan_eligible(nt, N) else "argmax_kernel",
                   "collective": ("one all_gather_into_tensor of the packed per-surface (max, index) pairs per step, asynchronous: it overlaps the next "
                                  "step's kernels (two buffers); all K exchanges complete inside the K timed brackets") if world > 1 else "none (1 GPU)",
                   "theta0_chain": chain, "bad_solves": nbad},
        "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": None if tps is None else tps * main_case["nsolve"], "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": solve_ms,
                     "share_of_step": float(t_solve.sum() / t_step.sum()),
                     "note": "FP64-pipe bound, not HBM bound (DESIGN.md section 3; see roofline_fp64): frac is the HBM fraction asked for; "
                             "kernel_ms = CUDA-event time of the solve call (coefficient prep + solver kernel incl. fused arg-max); "
                             "traffic = ncu dram bytes per launch of the solver kernel"},
        "roofline_fp64": rf64,
        "kernel_ms": {"geometry(K1 incl. pack+dPdrho)": float(t_geo.mean()), "solve(K2+K3+argmax)": solve_ms,
                      "collective": float(t_coll.mean()), "step": float(t_step.mean())},
        "gpu_launches": launches * args.steps,
        "step_ms": {"min": float(t_step.min()), "median": float(np.median(t_step)), "max": float(t_step.max())},
        "clocks": clocks, "wall_s_timed_region": wall,
    }
    if single:
        line["single_equilibrium"] = single
    if e2e:
        line["e2e"] = e2e
    if e2e_full:
        line["e2e_full_X"] = e2e_full
    if not args.no_cpu_baseline and world == 1:
        v, cores, sample, cw, kind_cpu = cpu_reference_rate(args.workload)
        line["cpu_baseline"] = {"value": v, "unit": "solves/s", "cores": cores, "kind": kind_cpu, "sample": sample}
    H.finish(line)


def run_salpha(H, args):
    torch = H.torch
    from ideal_ballooning_solver_b200 import engine, scan
    world, rank, dev = H.world, H.rank, H.dev
    _, shat, alpha, theta0, theta = workload_grids("salpha")
    N, h = len(theta), engine.grid_spacing(theta)
    lo, hi = scan.shard_range(len(shat), rank, world)               # N > 1: rows of the shat grid (total work fixed)
    sh_l = shat[lo:hi]
    S, A, T = np.meshgrid(sh_l, alpha, theta0, indexing="ij")
    prm = np.stack([S.ravel(), A.ravel(), T.ravel()], axis=1)       # (nsolve, 3), theta0 fastest
    nsolve = prm.shape[0]
    th_d = torch.from_numpy(theta).to(dev)

    def coefficients(p_d):
        # bishop_ball_s-alpha.py:30-45: Lambda = shat (th - th0) - alpha (sin th - sin th0); g = f = 1 + Lambda^2; c = alpha (cos + Lambda sin)
        sh, al, t0 = p_d[:, 0:1], p_d[:, 1:2], p_d[:, 2:3]
        L = sh * (th_d - t0) - al * (torch.sin(th_d) - torch.sin(t0))
        g = 1.0 + L * L
        return g, al * (torch.cos(th_d) + torch.sin(th_d) * L)

    prm_d = torch.from_numpy(prm).to(dev)
    g_d, c_d = coefficients(prm_d)
    rows_max = (len(shat) + world - 1) // world * len(alpha)
    cls_all = torch.zeros((world, rows_max), dtype=torch.uint8, device=dev)
    cls_send = torch.zeros((rows_max,), dtype=torch.uint8, device=dev)

    def step(t):
        rec(t, 0)
        sol = engine.solve_gcf_batch(g_d, c_d, g_d, h, want_X=True, want_dX=False, want_matrix=False, chain_len=len(theta0))
        rec(t, 1)
        # unstable <=> lambda_max > 0 for ANY of the theta0 (bishop_ball_s-alpha.py:282-289)
        cls = (sol.lam.reshape(-1, len(theta0)) > 0).any(dim=1)
        cls_send[: cls.numel()] = cls
        if world > 1:
            H.dist.all_gather_into_tensor(cls_all.view(-1), cls_send)
        rec(t, 2)
        return sol, cls

    sol, cls = step(None)
    torch.cuda.synchronize()
    nbad = int(np.count_nonzero((sol.info >> 16).cpu().numpy() & 3))
    mean_iters = float((sol.info & 0xFFFF).double().mean().item())
    total_s, stage, t_step, wall = H.timed(step, 2, keep_last=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        sol_l, cls_l = H.last_out
        dump_outputs(args.dump_outputs, {"gamma": sol_l.lam, "X": sol_l.X, "flags": sol_l.info >> 16, "unstable": cls_l})
    H.last_out = sol_l = None
    nsolve_all = len(shat) * len(alpha) * len(theta0)
    value = nsolve_all * args.steps / total_s
    clocks = H.clocks()
    e2e = None
    if not args.no_e2e:
        prm_p = torch.from_numpy(prm).pin_memory()
        lam_h = torch.empty(nsolve, dtype=torch.float64).pin_memory()
        cls_h = torch.empty(cls.numel(), dtype=torch.bool).pin_memory()

        def once():
            p_d = prm_p.to(dev, non_blocking=True)
            g, c = coefficients(p_d)
            s_ = engine.solve_gcf_batch(g, c, g, h, want_X=True, want_dX=False, want_matrix=False, chain_len=len(theta0))
            lam_h.copy_(s_.lam, non_blocking=True)
            cls_h.copy_((s_.lam.reshape(-1, len(theta0)) > 0).any(dim=1), non_blocking=True)
            torch.cuda.synchronize()
        once(); once()
        H.barrier()
        ke = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(ke):
            once()
        dt_e = H.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": nsolve_all * ke / dt_e, "unit": "solves/s", "h2d_bytes_per_step": int(prm.nbytes),
               "d2h_bytes_per_step": int(8 * nsolve + cls.numel()),
               "api": "engine.solve_gcf_batch on coefficients formed on the device from the pinned (shat, alpha, theta0) list; "
                      "lambda of every solve + the stability map copied back", "eigvec": "X of every solve written to HBM, not copied"}
    if rank != 0:
        return H.finish(None)
    peak, peak_src = load_peaks()
    solve_ms = float(stage[:, 0].mean())
    alg_bytes = 32.0 * N * nsolve
    achieved = alg_bytes / (solve_ms * 1e-3) / 1e9
    kname = "solve_kernel (K2+K3, team per solve)"
    line = {"metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": float(1e3 * total_s / args.steps), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic (analytic s-alpha coefficients)",
            "config": {"workload": describe("salpha"), "solves_per_step_per_gpu": nsolve, "l2": "flushed between timed steps (256 MB write)",
                       "eigvec": "X written to HBM for every solve", "mean_solver_iterations": mean_iters, "solver": kname,
                       "unstable_points": int(cls.sum().item()), "grid_points_per_gpu": int(cls.numel()), "bad_solves": nbad},
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": solve_ms,
                         "share_of_step": float(stage[:, 0].sum() / t_step.sum())},
            "roofline_fp64": fp64_rooflines(H, [(kname, N * nsolve * (22.0 * mean_iters + 40.0), solve_ms, "FMAs per solve = N x (22 x evaluations + 40)")]),
            "kernel_ms": {"solve(K2+K3)": solve_ms, "classify+collective": float(stage[:, 1].mean()), "step": float(t_step.mean())},
            "gpu_launches": 1 * args.steps, "step_ms": {"min": float(t_step.min()), "median": float(np.median(t_step)), "max": float(t_step.max())},
            "clocks": clocks, "wall_s_timed_region": wall}
    if e2e:
        line["e2e"] = e2e
    if not args.no_cpu_baseline and world == 1:
        v, cores, sample, cw, kind_cpu = cpu_reference_rate("salpha")
        line["cpu_baseline"] = {"value": v, "unit": "solves/s", "cores": cores, "kind": kind_cpu, "sample": sample}
    H.finish(line)


def run_adjoint(H, args):
    torch = H.torch
    from ideal_ballooning_solver_b200 import engine, synthetic, tables
    world, rank, dev = H.world, H.rank, H.dev
    npts = args.points
    kind, _, _, _, theta = workload_grids("adjoint")
    N, h, d = len(theta), engine.grid_spacing(theta), ADJOINT["del_alpha"]
    rng = np.random.default_rng(20261018 + 5 + 1000 * rank)
    s = rng.uniform(0.5, 0.95, npts); al = rng.uniform(0, np.pi, npts); t0 = rng.uniform(0, 0.5 * np.pi, npts)
    st = tables.RadialSplines(synthetic.make_equilibrium(kind, seed=1)).evaluate(s)          # one table set per point (i.i.d. s)
    dt = engine.DeviceTables.from_host(st, dev)
    alphas_h = np.stack([al - 0.5 * d, al, al + 0.5 * d], axis=1)                           # utils.py:1641-1646
    alphas = torch.from_numpy(alphas_h).to(dev)
    th_d, t0_d = torch.from_numpy(theta).to(dev), torch.from_numpy(t0).to(dev)
    grads = torch.zeros((world, npts, 2), dtype=torch.float64, device=dev)

    def step(t):
        rec(t, 0)
        geo = engine.geometry_batch(dt, alphas, th_d)
        rec(t, 1)
        val, grad, X, dX, info = engine.obj_w_grad_batch(geo.base, geo.dPdrho, t0_d, h, del_alpha=d, want_X=True)
        rec(t, 2)
        if world > 1:                    # the one exchange of this workload: gradients of every rank's points (16 B per point)
            H.dist.all_gather_into_tensor(grads.view(-1), grad.view(-1))
        rec(t, 3)
        return val, grad, info, X, dX

    val, grad, info = step(None)[:3]
    torch.cuda.synchronize()
    nbad = int(np.count_nonzero((info >> 16).cpu().numpy() & 3))
    mean_iters = float((info & 0xFFFF).double().mean().item())
    total_s, stage, t_step, wall = H.timed(step, 3, keep_last=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        val_l, grad_l, info_l, X_l, dX_l = H.last_out
        dump_outputs(args.dump_outputs, {"val": val_l, "grad": grad_l, "X": X_l, "dX": dX_l, "flags": info_l >> 16})
    H.last_out = X_l = dX_l = None
    value = world * npts * args.steps / total_s
    clocks = H.clocks()
    e2e = None
    if not args.no_e2e:
        import dataclasses
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        tm_p, tn_p, sc_p, al_p, t0_p = pin(st.tab_mn), pin(st.tab_nyq), pin(st.scal), pin(alphas_h), pin(t0)
        val_h, grad_h = torch.empty(npts, dtype=torch.float64).pin_memory(), torch.empty((npts, 2), dtype=torch.float64).pin_memory()

        def once():
            dt_e = dataclasses.replace(dt, tab_mn=tm_p.to(dev, non_blocking=True), tab_nyq=tn_p.to(dev, non_blocking=True),
                                       scal=sc_p.to(dev, non_blocking=True))
            geo = engine.geometry_batch(dt_e, al_p.to(dev, non_blocking=True), th_d)
            v, g, _, _, _ = engine.obj_w_grad_batch(geo.base, geo.dPdrho, t0_p.to(dev, non_blocking=True), h, del_alpha=d)
            val_h.copy_(v, non_blocking=True); grad_h.copy_(g, non_blocking=True)
            torch.cuda.synchronize()
        once()
        H.barrier()
        ke = 3
        tt = time.perf_counter()
        for _ in range(ke):
            once()
        dt_s = H.max_over_ranks(time.perf_counter() - tt)
        e2e = {"value": world * npts * ke / dt_s, "unit": "solves/s",
               "h2d_bytes_per_step": int(st.tab_mn.nbytes + st.tab_nyq.nbytes + st.scal.nbytes + alphas_h.nbytes + t0.nbytes),
               "d2h_bytes_per_step": int(24 * npts), "api": "engine.geometry_batch + engine.obj_w_grad_batch (ibs_geometry_batch, "
               "ibs_obj_w_grad_batch) on per-point Fourier tables uploaded from pinned host memory; (-lambda, gradient) of every point copied back",
               "eigvec": "X, dX of every solve formed in HBM (consumed by K4), not copied"}
    if rank != 0:
        return H.finish(None)
    peak, peak_src = load_peaks()
    solve_ms = float(stage[:, 1].mean())
    alg_bytes = (32.0 + 8.0) * N * npts + (3 * 8) * 8.0 * N * npts        # solver (g,c,f in, X, dX out) + K4 reading three lines of 8 base arrays
    achieved = alg_bytes / (solve_ms * 1e-3) / 1e9
    kname = "solve_kernel (K2+K3, team per solve) + obj_grad_kernel (K4)"
    fma_geo = (10.0 * len(st.xm) + 9.0 * len(st.xm_nyq)) * N * 3 * npts
    line = {"metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": float(1e3 * total_s / args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": describe("adjoint", points=npts), "solves_per_step_per_gpu": npts, "field_lines_per_step_per_gpu": 3 * npts,
                       "l2": "flushed between timed steps (256 MB write)", "eigvec": "X and dX written to HBM for every solve",
                       "mean_solver_iterations": mean_iters, "solver": kname,
                       "collective": "all_gather_into_tensor of the gradients (16 B per point)" if world > 1 else "none (1 GPU)",
                       "bad_solves": nbad, "grad_finite": bool(torch.isfinite(grad).all().item())},
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": solve_ms,
                         "share_of_step": float(stage[:, 1].sum() / t_step.sum()),
                         "note": "the step is dominated by K1 (three field lines per point, FP64-pipe bound: see roofline_fp64)"},
            "roofline_fp64": fp64_rooflines(H, [("geometry_kernel (K1)", fma_geo, float(stage[:, 0].mean()), "algorithmic FMAs per point = 10 mnmax + 9 mnmax_nyq; three field lines per (s, alpha, theta0) point")]),
            "kernel_ms": {"geometry(K1, 3 lines per point)": float(stage[:, 0].mean()), "solve+adjoint(K2+K3+K4)": solve_ms,
                          "collective": float(stage[:, 2].mean()), "step": float(t_step.mean())},
            "gpu_launches": 7 * args.steps,      # pack_mn, pack_nyq, geometry, dpdrho, centre_lines, solve, obj_grad
            "step_ms": {"min": float(t_step.min()), "median": float(np.median(t_step)), "max": float(t_step.max())},
            "clocks": clocks, "wall_s_timed_region": wall}
    if e2e:
        line["e2e"] = e2e
    if not args.no_cpu_baseline and world == 1:
        v, cores, sample, cw, kind_cpu = cpu_reference_rate("adjoint")
        line["cpu_baseline"] = {"value": v, "unit": "solves/s", "cores": cores, "kind": kind_cpu, "sample": sample}
    H.finish(line)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="d3d", choices=ALL_WORKLOADS)
    ap.add_argument("--equilibria", type=int, default=None,
                    help="independent equilibria batched per step per GPU (default 37 for d3d: 37 x 128 lines x 2 theta0 groups = 9472 items "
                         "= 8 full rounds of the 148 x 8 resident warps of the solver kernel; 1 for ncsx / hberg = the configs as stated)")
    ap.add_argument("--points", type=int, default=ADJOINT["points"], help="adjoint workload: (s, alpha, theta0) points per GPU")
    ap.add_argument("--strong", action="store_true", help="scan workloads: shard ONE batch of surfaces over the ranks (total work fixed)")
    ap.add_argument("--chain", type=int, default=-1, help="warm-start run length over theta0 (-1 = scan default, 1 = off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-full", action="store_true", help="skip the second end-to-end figure (X of every solve over PCIe)")
    ap.add_argument("--no-single", action="store_true", help="skip the single-equilibrium measurement of the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, float64, at most 64 MB: arrays "
                         "too large for that as a fixed seeded sample of their rows, indices in DIR/<name>_rows.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.equilibria is None:
        args.equilibria = 37 if args.workload == "d3d" else 1
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the GPU implementation")
        return run_reference_arm(args)
    H = Harness(args)
    if args.workload == "salpha":
        return run_salpha(H, args)
    if args.workload == "adjoint":
        return run_adjoint(H, args)
    return run_scan(H, args)


if __name__ == "__main__":
    main()
