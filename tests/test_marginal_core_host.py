"""CPU check of the marginal-stability lane code (csrc/ibs_marginal_core.cuh) through the g++ harness
tools/marginal_core_host.cpp: the same record preparation, sweeps, root finder and null-vector outputs the CUDA kernel runs,
against the LAPACK + brentq oracle (oracle/marginal_oracle.py).  The harness is test infrastructure, not a fallback."""
import os
import shutil
import sys

import numpy as np
import pytest

from helpers import s_alpha_base
from oracle import marginal_oracle as mo

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tools"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

FIXTURES = ["ncsx_wout_op", "synthetic_ncsx", "synthetic_d3d", "synthetic_hberg"]
THETA0 = np.array([0.0, np.pi / 8, np.pi / 4, 3 * np.pi / 8, np.pi / 2])
STABLE, NOT_CONVEX = 8, 16


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    import marginal_host_check as mhc
    return mhc, mhc.build(str(tmp_path_factory.mktemp("mch")))


@pytest.mark.parametrize("name", FIXTURES)
def test_kappa_star_matches_oracle(harness, golden, name):
    mhc, lib = harness
    D = golden(name)
    base, dP = mhc.fixture_lines(D)
    theta = D["theta"]
    nl, nt = base.shape[0], len(THETA0)
    R = mhc.solve(lib, base, dP, np.tile(THETA0, nl), theta[1] - theta[0], nth0=nt, want_X=False)
    assert np.all((R["info"] >> 16) == 0)
    sweeps = (R["info"] & 0xFFFF).mean()
    print(f"{name}: {sweeps:.2f} sweeps per solve")
    assert sweeps <= 10.0                          # measured 6.5 - 8.7 on the four fixtures
    for line in range(nl):
        for t, th0 in enumerate(THETA0):
            k = R["kappa"][line * nt + t]
            ks = mo.kappa_star(base[line], dP[line], theta, th0)
            assert abs(k - ks) <= 1e-9 * ks, (line, t, k, ks)
            # certificates: stable just below kappa*, unstable just above it
            rec = R["rec"][line]
            assert mhc.count_at(lib, rec, th0, k * (1 - 1e-8)) == 0
            assert mhc.count_at(lib, rec, th0, k * (1 + 1e-8)) >= 1


def test_null_vector_and_derivatives(harness, golden):
    mhc, lib = harness
    D = golden("synthetic_d3d")
    base, dP = mhc.fixture_lines(D)
    theta = D["theta"]
    th0 = np.array([0.0, np.pi / 4, 0.3, 1.2])
    nl, nt = base.shape[0], len(th0)
    R = mhc.solve(lib, base, dP, np.tile(th0, nl), theta[1] - theta[0], nth0=nt, want_X=True)
    for line in range(nl):
        for t in range(nt):
            s = line * nt + t
            k, X = R["kappa"][s], R["X"][s]
            assert X.min() >= 0.0 and X.max() == 1.0 and X[0] == 0.0 and X[-1] == 0.0
            dl = mo.dlam_dkappa(base[line], dP[line], theta, th0[t], k)
            dk = mo.dkappa_dtheta0(base[line], dP[line], theta, th0[t])
            assert abs(R["dlam_dkappa"][s] - dl) <= 1e-6 * abs(dl), (s, R["dlam_dkappa"][s], dl)
            assert abs(R["dkappa_dtheta0"][s] - dk) <= 1e-6 * max(abs(dk), k)      # (0 at theta0 = 0 on up-down symmetric lines), (s, R["dkappa_dtheta0"][s], dk)


def test_flags(harness, golden):
    mhc, lib = harness
    D = golden("synthetic_d3d")
    base, dP = mhc.fixture_lines(D)
    theta = D["theta"]
    h = theta[1] - theta[0]
    # dPdrho = 0: c = 0, never unstable
    R = mhc.solve(lib, base[:1], np.zeros(1), np.zeros(1), h, want_X=False)
    assert R["kappa"][0] == np.inf and (R["info"][0] >> 16) == STABLE and (R["info"][0] & 0xFFFF) == 0
    # kappa_max below kappa* (>= 1.9 on these lines)
    R = mhc.solve(lib, base, dP, np.zeros(len(dP)), h, nth0=1, kappa_max=0.5, want_X=False)
    assert np.all(R["kappa"] == np.inf) and np.all((R["info"] >> 16) == STABLE)
    # non-finite input
    bad = base[:1].copy()
    bad[0, 4, 100] = np.nan
    R = mhc.solve(lib, bad, dP[:1], np.zeros(1), h, want_X=False)
    assert np.isnan(R["kappa"][0]) and (R["info"][0] >> 16) == 2
    # s-alpha base arrays: cvdrift - gbdrift is not a pressure term and changes sign -> NOT_CONVEX
    th = np.linspace(-5 * np.pi, 5 * np.pi, 1025)
    b, dp = s_alpha_base(0.8, 0.6, th)
    R = mhc.solve(lib, b[None], np.array([dp]), np.zeros(1), th[1] - th[0], want_X=False)
    assert (R["info"][0] >> 16) & NOT_CONVEX
    assert np.isfinite(R["kappa"][0]) or (R["info"][0] >> 16) & STABLE
