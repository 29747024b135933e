#!/usr/bin/env python
"""Cost of long field lines in the team solver: solve_base_batch with line_of_solve (the team kernel; one CTA up to
N = 8194, a thread-block cluster of 2, 4 or 8 CTAs above) at a fixed grid spacing, and one scan.refine_maxima on NCSX
surfaces.  CUDA events, medians over repetitions in which all variants alternate.
    python tools/bench_long_lines.py [reps=5]
Prints one JSON line per measurement (ms per call, us per solve, ns per solve-point) and a last line with the device name
and power limit.  The variant "forced_C2" runs the same N = 8193 batch on clusters of 2 CTAs (IBS_TEAM_CLUSTER=2)."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ideal_ballooning_solver_b200 import engine, scan, synthetic, tables

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
H = 8 * np.pi / 4096                     # grid spacing of every solve batch: theta in +-4 pi at N = 4097
st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=1)).evaluate(np.linspace(0.5, 0.95, 4))
dt = engine.DeviceTables.from_host(st)
rng = np.random.default_rng(20261020)


def solve_case(N, nsolve):
    theta = H * (np.arange(N) - (N - 1) / 2)
    geo = engine.geometry_batch(dt, np.linspace(0.1, np.pi - 0.1, 4), theta)     # 16 lines
    nline = geo.base.numel() // (engine.NBASE * N)
    line = torch.from_numpy(rng.integers(0, nline, nsolve).astype(np.int32)).cuda()
    th0 = torch.from_numpy(rng.uniform(0.0, 0.5 * np.pi, nsolve)).cuda()
    h = engine.grid_spacing(theta)
    return lambda: engine.solve_base_batch(geo.base, geo.dPdrho, th0, h, line_of_solve=line, want_dX=False, want_matrix=False)


def forced(fn, C):
    def run():
        os.environ["IBS_TEAM_CLUSTER"] = str(C)
        try:
            return fn()
        finally:
            del os.environ["IBS_TEAM_CLUSTER"]
    return run


variants = {}
for nsolve in (64, 4096):
    for N in (4097, 8193, 16385, 32769, 65537):
        variants[("solve", N, nsolve, "auto")] = solve_case(N, nsolve)
    variants[("solve", 8193, nsolve, "forced_C2")] = forced(variants[("solve", 8193, nsolve, "auto")], 2)
st64 = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=1)).evaluate(np.linspace(0.5, 0.95, 64))
dt64 = engine.DeviceTables.from_host(st64)
a_g, t_g = rng.uniform(0.2, 2.8, 64), rng.uniform(0.0, 1.4, 64)
for N in (8193, 16385):
    theta = np.linspace(-8 * np.pi, 8 * np.pi, N)
    variants[("refine", N, 64, "auto")] = lambda theta=theta: scan.refine_maxima(dt64, a_g, t_g, theta)

for fn in variants.values():                      # warm-up: module load, memory pool, per-device attributes
    fn()
torch.cuda.synchronize()
times = {k: [] for k in variants}
for _ in range(reps):
    for k, fn in variants.items():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times[k].append(e0.elapsed_time(e1))
for (what, N, nsolve, mode), v in times.items():
    ms = float(np.median(v))
    cta = 1 if (N - 2 <= 8192 and mode == "auto") else (2 if mode == "forced_C2" else next(c for c in (2, 4, 8) if N - 2 <= c * 8192))
    row = {"what": what, "N": N, "nsolve": nsolve, "mode": mode, "ctas_per_solve": cta if what == "solve" else None,
           "ms": ms, "ms_min": float(np.min(v)), "us_per_solve": 1e3 * ms / nsolve, "ns_per_solve_point": 1e6 * ms / (nsolve * N)}
    print(json.dumps(row))
dev = torch.cuda.current_device()
try:
    smi = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError):
    smi = "unknown"
print(json.dumps({"device": torch.cuda.get_device_name(dev), "power_limit": smi, "reps": reps, "h": H}))
