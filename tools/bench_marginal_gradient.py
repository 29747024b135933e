#!/usr/bin/env python
"""Cost of the kappa* path for an optimiser against the growth-rate path, on 64 NCSX-like surfaces at nl = 2049 (the
configuration of tools/bench_scalar_gradient.py), CUDA events, variants alternated in every repetition, medians:
  gradient:   scan.marginal_gradient(..., scalars=True) against scan.table_gradient(..., scalars=True) at the same points;
  refinement: scan.refine_marginal against scan.refine_maxima(alpha_derivative="exact"), each from its own coarse optimum on
              the reference's 24 x 15 grid (marginal_scan / coarse_scan), with the rounds each takes.
    python tools/bench_marginal_gradient.py [reps=10] [OUT.json]
Prints one JSON object with the device name and power limit beside the times (and writes it to OUT.json when given)."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ideal_ballooning_solver_b200 import engine, scan, synthetic, tables

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
out_path = sys.argv[2] if len(sys.argv) > 2 else None
ns, nl = 64, 2049
st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=1)).evaluate(np.linspace(0.5, 0.95, ns))
theta = np.linspace(-4 * np.pi, 4 * np.pi, nl)
rng = np.random.default_rng(20261018)
a_star, t_star = rng.uniform(0, np.pi, ns), rng.uniform(0, 0.5 * np.pi, ns)
dt = engine.DeviceTables.from_host(st)
alpha_grid, theta0_grid = np.linspace(0, np.pi, scan.NALPHA_GUESS), np.linspace(0, 0.5 * np.pi, scan.NTHETA0_GUESS)
ms = scan.marginal_scan(dt, alpha_grid, theta0_grid, theta)
cs = scan.coarse_scan(dt, alpha_grid, theta0_grid, theta)
ka, kt = ms.alpha_crit.cpu().numpy(), ms.theta0_crit.cpu().numpy()
ga, gt = cs.alpha_guess.cpu().numpy(), cs.theta0_guess.cpu().numpy()
rounds = {}


def refine_marginal():
    rounds["refine_marginal"] = scan.refine_marginal(dt, ka, kt, theta).nbatches


def refine_maxima():
    rounds["refine_maxima_exact"] = scan.refine_maxima(dt, ga, gt, theta, alpha_derivative="exact").nbatches


variants = {
    "marginal_gradient_scalars": lambda: scan.marginal_gradient(dt, a_star, t_star, theta, scalars=True),
    "table_gradient_scalars": lambda: scan.table_gradient(dt, a_star, t_star, theta, scalars=True),
    "refine_marginal": refine_marginal,
    "refine_maxima_exact": refine_maxima,
}
for fn in variants.values():                      # warm-up: module load, memory pool
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
dev = torch.cuda.current_device()
try:
    smi = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError):
    smi = "unknown"
kmin = ms.kappa_min.cpu().numpy()
out = {"device": torch.cuda.get_device_name(dev), "power_limit": smi, "ns": ns, "nl": nl, "reps": reps,
       "finite_kappa_min": int(np.isfinite(kmin).sum()), "rounds": rounds}
for k, v in times.items():
    out[k + "_ms"] = float(np.median(v))
    out[k + "_ms_min"] = float(np.min(v))
out["marginal_over_table_gradient"] = out["marginal_gradient_scalars_ms"] / out["table_gradient_scalars_ms"]
out["refine_marginal_over_refine_maxima"] = out["refine_marginal_ms"] / out["refine_maxima_exact_ms"]
print(json.dumps(out))
if out_path:
    with open(out_path, "w") as f:
        json.dump(out, f, indent=1)
