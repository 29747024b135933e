"""Drive the CPU harness of the scan solver's lane code (tools/scan_core_host.cpp) on a golden fixture and compare
with the oracle (LAPACK lambda_max route).  Test tooling only.

    python tools/scan_host_check.py [fixture] [nth0] [--sigma]
"""
import ctypes
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
from oracle import ballooning_oracle as bo  # noqa: E402

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
BASE_NAMES = ["bmag", "gradpar_theta_pest", "cvdrift", "cvdrift0", "gds2", "gds21", "gds22", "gbdrift"]


def build(outdir="/tmp/sch"):
    """Compile the harness (tools/scan2_core_host.cpp: it includes scan_core_host.cpp, so one library carries the lane code
    of both kernels: scan_host_solve = two chains per lane, scan2_host_solve = one chain per lane)."""
    os.makedirs(outdir, exist_ok=True)
    so = os.path.join(outdir, "scan_core_host.so")
    srcs = [os.path.join(ROOT, "tools", n) for n in ("scan2_core_host.cpp", "scan_core_host.cpp")]
    hdrs = [os.path.join(ROOT, "ideal-ballooning-solver_b200", "csrc", n) for n in ("ibs_scan_core.cuh", "ibs_scan2_core.cuh")]
    if not os.path.isfile(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in srcs + hdrs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so, srcs[0]])
    lib = ctypes.CDLL(so)
    dp = ctypes.POINTER(ctypes.c_double)
    ip = ctypes.POINTER(ctypes.c_int)
    lib.scan_host_rows_total.restype = ctypes.c_int
    lib.scan_host_num_levels.restype = ctypes.c_int
    lib.scan_host_prep.argtypes = [dp, dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, dp, dp]
    lib.scan_host_solve.restype = ctypes.c_long
    lib.scan_host_last_cost.restype = ctypes.c_double
    lib.scan_host_solve.argtypes = [dp, dp, dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, dp, dp, dp, dp, ip]
    lib.scan2_host_solve.restype = ctypes.c_long
    lib.scan2_host_solve.argtypes = lib.scan_host_solve.argtypes
    lib.scan2_host_size_ok.restype = ctypes.c_int
    return lib


def _p(a, t=ctypes.c_double):
    return a.ctypes.data_as(ctypes.POINTER(t)) if a is not None else None


def host_scan_solve(lib, base, dPdrho, theta0, h, sigma=None, want_X=True, want_dX=True, kernel="scan"):
    """base (nline, 8, N), dPdrho (nline,), theta0 (nline, nth0) -> dict of results from the CPU harness.
    kernel = "scan": lane code of scan_solve_kernel (two chains per lane); "scan2": of scan2_solve_kernel (one chain per lane)."""
    base = np.ascontiguousarray(base, dtype=np.float64)
    nline, _, N = base.shape
    theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
    nth0 = theta0.shape[1]
    rows_total = lib.scan_host_rows_total(N)
    poly = np.zeros((nline, rows_total, 6))
    bounds = np.zeros((nline, 2))
    dP = np.ascontiguousarray(dPdrho, dtype=np.float64)
    lib.scan_host_prep(_p(base), _p(dP), _p(theta0), nline, nth0, N, float(h), _p(poly), _p(bounds))
    n = nline * nth0
    lam = np.zeros(n); lm = np.zeros(n)
    X = np.full((n, N), np.nan) if want_X else None
    dX = np.full((n, N), np.nan) if want_dX else None
    info = np.zeros(n, dtype=np.int32)
    sg = np.ascontiguousarray(sigma, dtype=np.float64) if sigma is not None else None
    passes = (lib.scan2_host_solve if kernel == "scan2" else lib.scan_host_solve)(_p(poly), _p(bounds), _p(theta0), _p(sg), nline, nth0, N, float(h), _p(lam), _p(lm), _p(X), _p(dX),
                                 _p(info, ctypes.c_int))
    return dict(lam=lam.reshape(nline, nth0), lam_matrix=lm.reshape(nline, nth0), X=X, dX=dX, info=info.reshape(nline, nth0),
                passes=passes, bounds=bounds, poly=poly, cost=lib.scan_host_last_cost())


def oracle_solve(D, i, j, th0, method="lambda_max"):
    cv = D["geo_cvdrift"][i, j] + th0 * D["geo_cvdrift0"][i, j]
    gd = D["geo_gds2"][i, j] + 2 * th0 * D["geo_gds21"][i, j] + th0 ** 2 * D["geo_gds22"][i, j]
    info = {}
    gam, X, dX, *_ = bo.gamma_ball_full(D["dPdrho"][i, j], D["theta"], D["geo_bmag"][i, j], D["geo_gradpar_theta_pest"][i, j], cv, gd,
                                        method=method, info=info)
    s = np.sign(X[np.argmax(np.abs(X))])
    return gam, X * s, dX * s, info


def main():
    fx = sys.argv[1] if len(sys.argv) > 1 else "synthetic_d3d"
    nth0 = int(sys.argv[2]) if len(sys.argv) > 2 else 8
    D = np.load(os.path.join(ROOT, "tests", "golden", f"{fx}.npz"))
    lib = build()
    ns, na = D["geo_bmag"].shape[:2]
    base = np.stack([D["geo_" + n] for n in BASE_NAMES], axis=2).reshape(ns * na, 8, -1)
    dP = D["dPdrho"].reshape(-1)
    th0 = np.tile(np.linspace(0, np.pi / 2, nth0), (ns * na, 1))
    theta = D["theta"]
    h = theta[1] - theta[0]
    sigma = np.full(th0.size, 1.0) if "--sigma" in sys.argv else None
    R = host_scan_solve(lib, base, dP, th0, h, sigma=sigma)
    N = base.shape[2]
    print("levels", lib.scan_host_num_levels(N), "passes/solve", R["passes"] / th0.size, "fine-equivalent passes/solve", R["cost"] / th0.size, "info its", (R["info"] & 0xffff).mean(),
          "flags", np.unique(R["info"] >> 16))
    el = ex = ed = 0.0
    for line in range(ns * na):
        i, j = divmod(line, na)
        for t in range(nth0):
            gam, X, dX, info = oracle_solve(D, i, j, th0[line, t])
            s = line * nth0 + t
            el = max(el, abs(R["lam"][line, t] - gam) / abs(gam))
            ex = max(ex, np.max(np.abs(R["X"][s] - X)))
            ed = max(ed, np.max(np.abs(R["dX"][s] - dX)) / np.max(np.abs(dX)))
    print(f"lam rel err {el:.2e}   X abs err {ex:.2e}   dX rel-to-max err {ed:.2e}")


if __name__ == "__main__":
    main()
