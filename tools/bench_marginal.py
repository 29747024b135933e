"""Time engine.marginal_batch (prep + solve kernels) on the bench's scan batches, and in the same process the coarse scan's
solve leg (engine.scan_solve_argmax: K2+K3 with the fused arg-max) on the same field lines.  K1 runs once, untimed.

    python tools/bench_marginal.py [--reps R] [--out profiles/marginal_r03.json]

Records the device name and power limit beside the numbers.  Needs a GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def run(name, equilibria, reps):
    import torch
    import bench
    from ideal_ballooning_solver_b200 import engine, scan
    st, alpha, theta0, theta = bench.build_tables(name, equilibria, seed0=0)
    dt = engine.DeviceTables.from_host(st)
    geo = engine.geometry_batch(dt, alpha, theta)
    ns, na, nt = dt.ns, len(alpha), len(theta0)
    h = engine.grid_spacing(theta)
    th0 = torch.from_numpy(theta0).cuda().repeat(ns * na)
    res = {}
    m = engine.marginal_batch(geo.base, geo.dPdrho, th0, h, nth0=nt)
    torch.cuda.synchronize()
    out = dict(workload=name, equilibria=equilibria, solves=int(th0.numel()), N=len(theta),
               sweeps_mean=float(m.sweeps.double().mean().item()), sweeps_max=int(m.sweeps.max().item()),
               flags=sorted(set(int(v) for v in m.flags.unique().cpu().numpy())),
               kappa_min=float(m.kappa.min().item()), unstable_fraction=float((m.kappa < 1).double().mean().item()))
    # alternate the two legs so that both see the same clocks
    tm, ts = [], []
    for _ in range(3):
        tm.append(timed(lambda: engine.marginal_batch(geo.base, geo.dPdrho, th0, h, nth0=nt), reps))
        ts.append(timed(lambda: engine.scan_solve_argmax(geo.base, geo.dPdrho, th0, h, nt, na, chain_len=scan.chain_length(nt)), reps))
    out["marginal_ms_median"] = float(np.median([t[0] for t in tm]))
    out["marginal_ms_min"] = float(min(t[1] for t in tm))
    out["solve_leg_ms_median"] = float(np.median([t[0] for t in ts]))
    out["solve_leg_ms_min"] = float(min(t[1] for t in ts))
    out["ratio_median"] = out["marginal_ms_median"] / out["solve_leg_ms_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    dev = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    rows = [run("d3d", 37, args.reps), run("ncsx", 1, args.reps)]
    result = dict(device=dev, power_limit_and_max_sm_clock=pl, results=rows)
    print(json.dumps(result, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
