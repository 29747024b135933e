#!/usr/bin/env python
"""Cost of the scalar gradients: scan.table_gradient(..., scalars=True) against scalars=False, and the reverse-mode K1 call
alone (ibs_geometry_adjoint_scal against ibs_geometry_adjoint), for NCSX-like surfaces, CUDA events, the two variants
alternated in every repetition.
    python tools/bench_scalar_gradient.py [ns=64] [nl=2049] [reps=20]
Prints one JSON line with the device name and power limit beside the times (ms, median over reps)."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ideal_ballooning_solver_b200 import engine, scan, synthetic, tables

ns = int(sys.argv[1]) if len(sys.argv) > 1 else 64
nl = int(sys.argv[2]) if len(sys.argv) > 2 else 2049
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 20
st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=1)).evaluate(np.linspace(0.5, 0.95, ns))
theta = np.linspace(-4 * np.pi, 4 * np.pi, nl)
rng = np.random.default_rng(20261018)
a_star, t_star = rng.uniform(0, np.pi, ns), rng.uniform(0, 0.5 * np.pi, ns)
dt = engine.DeviceTables.from_host(st)

# inputs of the reverse-mode call, formed as table_gradient forms them
a = torch.from_numpy(a_star[:, None].copy()).cuda()
t0 = torch.from_numpy(t_star.copy()).cuda()
geo = engine.geometry_batch(dt, a, theta)
sol = engine.solve_base_batch(geo.base, geo.dPdrho, t0, engine.grid_spacing(theta), nth0=1, want_dX=True, want_matrix=False,
                              want_gcf=True)
sg, sc, sf = engine.adjoint_sensitivities(sol.lam, sol.X, sol.dX, sol.f)
dP = geo.dPdrho.reshape(-1)
Q = (sc * sol.c).sum(dim=1) / (-dP)
adj_args = (dt, a.reshape(-1), theta, t0, dP, sg, sc, sf, Q)

variants = {
    "table_gradient": lambda: scan.table_gradient(dt, a_star, t_star, theta),
    "table_gradient_scalars": lambda: scan.table_gradient(dt, a_star, t_star, theta, scalars=True),
    "geometry_adjoint": lambda: engine.geometry_adjoint(*adj_args),
    "geometry_adjoint_scal": lambda: engine.geometry_adjoint(*adj_args, want_scalars=True),
}
for fn in variants.values():                      # warm-up: module load, memory pool
    for _ in range(2):
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
out = {"device": torch.cuda.get_device_name(dev), "power_limit": smi, "ns": ns, "nl": nl, "reps": reps,
       "mnmax": len(st.xm), "mnmax_nyq": len(st.xm_nyq)}
for k, v in times.items():
    out[k + "_ms"] = float(np.median(v))
    out[k + "_ms_min"] = float(np.min(v))
out["table_gradient_scalars_over_plain"] = out["table_gradient_scalars_ms"] / out["table_gradient_ms"]
out["geometry_adjoint_scal_over_plain"] = out["geometry_adjoint_scal_ms"] / out["geometry_adjoint_ms"]
print(json.dumps(out))
