"""Drive the CPU harness of the marginal-stability lane code (tools/marginal_core_host.cpp) on a golden fixture and compare
kappa* with the oracle (oracle/marginal_oracle.py).  Test tooling only.

    python tools/marginal_host_check.py [fixture]
"""
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from oracle import marginal_oracle as mo  # noqa: E402

BASE_NAMES = ["bmag", "gradpar_theta_pest", "cvdrift", "cvdrift0", "gds2", "gds21", "gds22", "gbdrift"]
MREC = 6


def build(outdir="/tmp/mch"):
    os.makedirs(outdir, exist_ok=True)
    so = os.path.join(outdir, "marginal_core_host.so")
    src = os.path.join(ROOT, "tools", "marginal_core_host.cpp")
    hdrs = [os.path.join(ROOT, "ideal-ballooning-solver_b200", "csrc", n) for n in ("ibs_scan_core.cuh", "ibs_marginal_core.cuh")]
    if not os.path.isfile(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in [src] + hdrs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so, src])
    lib = ctypes.CDLL(so)
    v, d, i = ctypes.c_void_p, ctypes.c_double, ctypes.c_int
    lib.marginal_host_prep.argtypes = [v, v, i, i, d, v, v]
    lib.marginal_host_solve.argtypes = [v, v, v, v, v, v, i, i, i, d, d, d, v, v, v, v, v]
    lib.marginal_host_sweep.argtypes = [v, i, d, d, ctypes.POINTER(d)]
    lib.marginal_host_sweep.restype = i
    lib.marginal_host_tangent.argtypes = [v, v, v, v, v, v, i, i, i, d, v, v, v]
    lib.marginal_host_sensitivities.argtypes = [v, v, v, v, i, i, i, d, v, v, v, v]
    return lib


def _p(a):
    return None if a is None else a.ctypes.data


def prep(lib, base, dPdrho, h):
    base = np.ascontiguousarray(base, dtype=np.float64)
    nline, _, N = base.shape
    rec = np.zeros((nline, N, MREC))
    flags = np.zeros(nline, dtype=np.int32)
    lib.marginal_host_prep(_p(base), _p(np.ascontiguousarray(dPdrho, dtype=np.float64)), nline, N, float(h), _p(rec), _p(flags))
    return rec, flags


def solve(lib, base, dPdrho, theta0, h, nth0=None, line_of_solve=None, kappa_max=1e3, rtol=1e-12, want_X=True):
    """base (nline, 8, N), dPdrho (nline,), theta0 (nsolve,) -> dict of results of the lane code."""
    base = np.ascontiguousarray(base, dtype=np.float64)
    dP = np.ascontiguousarray(dPdrho, dtype=np.float64)
    N = base.shape[2]
    rec, flags = prep(lib, base, dP, h)
    th0 = np.ascontiguousarray(theta0, dtype=np.float64).reshape(-1)
    n = th0.size
    los = None if line_of_solve is None else np.ascontiguousarray(line_of_solve, dtype=np.int32)
    kappa, dl, dk = np.zeros(n), np.zeros(n), np.zeros(n)
    X = np.zeros((n, N)) if want_X else None
    info = np.zeros(n, dtype=np.int32)
    lib.marginal_host_solve(_p(rec), _p(base), _p(dP), _p(flags), _p(th0), _p(los), int(nth0 or 1), n, N, float(h),
                            float(kappa_max), float(rtol), _p(kappa), _p(dl) if want_X else None, _p(dk) if want_X else None,
                            _p(X), _p(info))
    return dict(kappa=kappa, dlam_dkappa=dl, dkappa_dtheta0=dk, X=X, info=info, rec=rec, line_flags=flags)


def tangent(lib, base, dbase, dPdrho, ddPdrho, theta0, h, kappa, X, nth0=1):
    """d kappa* / d alpha of each solve along (dbase, ddPdrho) at (kappa, X) as ``solve`` returns them (scan-shaped batch)."""
    c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    base, dbase, dP, ddP, th0, kappa, X = (c(a) for a in (base, dbase, dPdrho, ddPdrho, theta0, kappa, X))
    out = np.zeros(th0.size)
    lib.marginal_host_tangent(_p(base), _p(dbase), _p(dP), _p(ddP), _p(th0), None, int(nth0), th0.size, base.shape[-1], float(h),
                              _p(kappa), _p(X), _p(out))
    return out


def sensitivities(lib, base, dPdrho, theta0, h, kappa, X, nth0=1):
    """(d kappa* / d g, d kappa* / d c) per point, each (nsolve, N)."""
    c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    base, dP, th0, kappa, X = (c(a) for a in (base, dPdrho, theta0, kappa, X))
    dg, dc = np.zeros_like(X), np.zeros_like(X)
    lib.marginal_host_sensitivities(_p(base), _p(dP), _p(th0), None, int(nth0), th0.size, base.shape[-1], float(h), _p(kappa), _p(X),
                                    _p(dg), _p(dc))
    return dg, dc


def count_at(lib, rec_line, theta0, kappa):
    phi = ctypes.c_double(0.0)
    return lib.marginal_host_sweep(_p(np.ascontiguousarray(rec_line)), rec_line.shape[0], float(theta0), float(kappa), ctypes.byref(phi))


def fixture_lines(D):
    ns, na = D["geo_bmag"].shape[:2]
    base = np.stack([D["geo_" + n] for n in BASE_NAMES], axis=2).reshape(ns * na, 8, -1)
    return base, D["dPdrho"].reshape(-1)


def main():
    fx = sys.argv[1] if len(sys.argv) > 1 else "synthetic_d3d"
    D = np.load(os.path.join(ROOT, "tests", "golden", f"{fx}.npz"))
    lib = build()
    base, dP = fixture_lines(D)
    theta = D["theta"]
    h = theta[1] - theta[0]
    th0s = np.array([0, np.pi / 8, np.pi / 4, 3 * np.pi / 8, np.pi / 2])
    nl = base.shape[0]
    R = solve(lib, base, dP, np.tile(th0s, nl), h, nth0=len(th0s))
    print("sweeps/solve", (R["info"] & 0xFFFF).mean(), "max", (R["info"] & 0xFFFF).max(), "flags", np.unique(R["info"] >> 16))
    err = 0.0
    for line in range(nl):
        for t, th0 in enumerate(th0s):
            ks = mo.kappa_star(base[line], dP[line], theta, th0)
            k = R["kappa"][line * len(th0s) + t]
            err = max(err, abs(k - ks) / ks)
            print(line, t, k, ks, (R["info"][line * len(th0s) + t] & 0xFFFF))
    print(f"kappa* rel err {err:.2e}")


if __name__ == "__main__":
    main()
