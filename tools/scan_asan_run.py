import sys, os, ctypes, numpy as np
sys.path.insert(0, "/root/repo"); sys.path.insert(0, "/root/repo/tools"); sys.path.insert(0, "/root/repo/tests")
import scan_host_check as shc
from helpers import s_alpha_base
# use the sanitised build
shc.build = lambda outdir=None: None
lib = ctypes.CDLL(os.environ.get("SCAN_ASAN_SO", "/tmp/sch_asan/scan_core_host.so"))
dp = ctypes.POINTER(ctypes.c_double); ip = ctypes.POINTER(ctypes.c_int)
lib.scan_host_rows_total.restype = ctypes.c_int; lib.scan_host_num_levels.restype = ctypes.c_int
lib.scan_host_prep.argtypes = [dp, dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, dp, dp]
lib.scan_host_solve.restype = ctypes.c_long; lib.scan_host_last_cost.restype = ctypes.c_double
lib.scan_host_solve.argtypes = [dp, dp, dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, dp, dp, dp, dp, ip]
lib.scan2_host_solve.restype = ctypes.c_long; lib.scan2_host_solve.argtypes = lib.scan_host_solve.argtypes
lib.scan2_host_size_ok.restype = ctypes.c_int
for n in (65, 129, 257, 969, 1025, 2049):
    theta = np.linspace(-6 * np.pi, 6 * np.pi, n)
    for th0max in (1.0, 15.0):
        th0 = np.linspace(0.0, th0max, 5)
        base, dP = s_alpha_base(0.8, 0.9, theta)
        R = shc.host_scan_solve(lib, base[None], np.array([dP]), th0[None], theta[1] - theta[0], sigma=np.full(5, 1.0))
        assert np.all(np.isfinite(R["lam"])), (n, th0max)
        if lib.scan2_host_size_ok(n):          # the lane-per-chain code: several lines, so that the warm-start records are read and written
            th0w = np.linspace(0.0, th0max, 20)
            bases = np.stack([s_alpha_base(0.8 + 0.01 * q, 0.9, theta)[0] for q in range(3)])
            dPs = np.array([s_alpha_base(0.8 + 0.01 * q, 0.9, theta)[1] for q in range(3)])
            R = shc.host_scan_solve(lib, bases, dPs, np.tile(th0w, (3, 1)), theta[1] - theta[0], sigma=np.full(60, 1.0), kernel="scan2")
            assert np.all(np.isfinite(R["lam"])), (n, th0max, "scan2")
D = np.load("/root/repo/tests/golden/synthetic_ncsx.npz")
base = np.stack([D["geo_" + k] for k in shc.BASE_NAMES], axis=2).reshape(-1, 8, len(D["theta"])).copy()
base[1, 4, 100] = np.nan
R = shc.host_scan_solve(lib, base, D["dPdrho"].reshape(-1), np.tile(np.linspace(0, 1.5, 4), (base.shape[0], 1)), D["theta"][1] - D["theta"][0])
R2 = shc.host_scan_solve(lib, base[:, :, :1009].copy(), D["dPdrho"].reshape(-1), np.tile(np.linspace(0, 1.5, 4), (base.shape[0], 1)), D["theta"][1] - D["theta"][0],
                         kernel="scan2") if lib.scan2_host_size_ok(1009) else None
print("asan run finished; flags", np.unique(R["info"] >> 16), None if R2 is None else np.unique(R2["info"] >> 16))
