#!/usr/bin/env python
"""The alpha-derivative of the growth rate two ways, timed in one process with CUDA events, alternating the two forms, medians:
  "fd":    K1 on three field lines per point (alpha -+ 0.002) -> ibs_obj_w_grad_batch (central difference, utils.py:1707-1725);
  "exact": K1 + its alpha-tangent on one line per point -> ibs_obj_w_grad_tangent_batch.
Workloads: K1 alone and the whole obj_w_grad evaluation on the adjoint configuration (NCSX-like tables, N = 1025, (s, alpha,
theta0) i.i.d. uniform with the bench's seeds) at 32 768 and 131 072 points; refine_maxima on 64 NCSX surfaces at N = 2049
and 8193.  Prints one JSON object with the card name and power limit (and writes it to OUT when given).
    python tools/bench_alpha_tangent.py [reps=7] [OUT]"""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ideal_ballooning_solver_b200 import engine, scan, synthetic, tables

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
D = 0.004


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record(); b.synchronize()
    return a.elapsed_time(b)


def alternate(fns, n):
    """median ms of each of fns, run alternately n times after one warm-up each"""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    t = {k: [] for k in fns}
    for _ in range(n):
        for k, f in fns.items():
            t[k].append(timed(f))
    return {k: float(np.median(v)) for k, v in t.items()}


def adjoint_config(npts):
    rng = np.random.default_rng(20261018 + 5)
    s = rng.uniform(0.5, 0.95, npts); al = rng.uniform(0, np.pi, npts); t0 = rng.uniform(0, 0.5 * np.pi, npts)
    theta = np.linspace(-4 * np.pi, 4 * np.pi, 1025)
    dt = engine.DeviceTables.from_host(tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=1)).evaluate(s))
    alphas3 = torch.from_numpy(np.stack([al - 0.5 * D, al, al + 0.5 * D], axis=1)).cuda()
    alpha1 = torch.from_numpy(al[:, None].copy()).cuda()
    th, t0d, h = torch.from_numpy(theta).cuda(), torch.from_numpy(t0).cuda(), engine.grid_spacing(theta)

    def k1_fd():
        return engine.geometry_batch(dt, alphas3, th)

    def k1_exact():
        return engine.geometry_tangent_batch(dt, alpha1, th)

    def owg_fd():
        g = k1_fd()
        return engine.obj_w_grad_batch(g.base, g.dPdrho, t0d, h, del_alpha=D, want_X=True)

    def owg_exact():
        g = k1_exact()
        return engine.obj_w_grad_tangent_batch(g.base, g.dbase, g.dPdrho, g.ddPdrho, t0d, h, want_X=True)

    k1_one = lambda: engine.geometry_batch(dt, alpha1, th)
    r = {"points": npts, "N": 1025}
    r.update({"K1_" + k + "_ms": v for k, v in alternate({"three_lines": k1_fd, "tangent_one_line": k1_exact, "one_line": k1_one},
                                                           reps).items()})
    r.update({"obj_w_grad_" + k + "_ms": v for k, v in alternate({"fd": owg_fd, "exact": owg_exact}, reps).items()})
    r["K1_tangent_over_one_line"] = r["K1_tangent_one_line_ms"] / r["K1_one_line_ms"]
    r["K1_tangent_over_three_lines"] = r["K1_tangent_one_line_ms"] / r["K1_three_lines_ms"]
    r["obj_w_grad_exact_over_fd"] = r["obj_w_grad_exact_ms"] / r["obj_w_grad_fd_ms"]
    g_fd, g_ex = owg_fd()[1][:, 0], owg_exact()[1][:, 0]
    r["abs_fd_minus_exact_over_max_exact"] = {"max": float(((g_fd - g_ex).abs().max() / g_ex.abs().max()).item()),
                                              "median": float(((g_fd - g_ex).abs().median() / g_ex.abs().max()).item())}
    return r


def refine_config(nl):
    st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=4)).evaluate(np.linspace(0.5, 0.95, 64))
    theta = np.linspace(-4 * np.pi, 4 * np.pi, nl)
    dt = engine.DeviceTables.from_host(st)
    res = scan.coarse_scan(dt, np.linspace(0, np.pi, 6), np.linspace(0, 0.5 * np.pi, 5), theta)
    a0, t0 = res.alpha_guess.clone(), res.theta0_guess.clone()
    out = {}
    fns = {k: (lambda k=k: out.__setitem__(k, scan.refine_maxima(dt, a0, t0, theta, alpha_derivative=k))) for k in ("fd", "exact")}
    r = {"surfaces": 64, "N": nl}
    r.update({"refine_" + k + "_ms": v for k, v in alternate(fns, max(3, reps // 2)).items()})
    for k in ("fd", "exact"):
        r["rounds_" + k] = int(out[k].nbatches)
        r["all_success_" + k] = bool(np.all(out[k].success))
    r["refine_exact_over_fd"] = r["refine_exact_ms"] / r["refine_fd_ms"]
    r["max_rel_fun_diff"] = float(np.max(np.abs(out["exact"].fun - out["fd"].fun) / np.abs(out["fd"].fun)))
    return r


t_start = time.time()
result = {"card": card(), "reps": reps, "adjoint": [adjoint_config(n) for n in (32768, 131072)],
          "refine": [refine_config(nl) for nl in (2049, 8193)]}
result["wall_s"] = time.time() - t_start
line = json.dumps(result)
print(line)
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as f:
        f.write(line + "\n")
