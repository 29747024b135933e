"""CPU check of the first-order response of kappa* at the null vector (csrc/ibs_marginal_core.cuh: record_tangent, point_forms,
point_sensitivities) through the g++ harness tools/marginal_core_host.cpp, against the LAPACK + brentq oracle: the alpha-tangent
form is a directional derivative of kappa*, the per-point sensitivities are the derivatives of kappa* with respect to the
pencil's coefficients, and they satisfy the scale identity of a null vector."""
import os
import shutil
import sys

import numpy as np
import pytest
from scipy.linalg import eigvalsh_tridiagonal
from scipy.optimize import brentq

from oracle import ballooning_oracle as bo
from oracle import marginal_oracle as mo

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tools"))

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")

FIXTURES = ["ncsx_wout_op", "synthetic_ncsx", "synthetic_d3d", "synthetic_hberg"]
THETA0 = np.array([0.0, 0.4, 1.1])
BMAG, GRADPAR, CVDRIFT, CVDRIFT0, GDS2, GDS21, GDS22, GBDRIFT = range(8)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    import marginal_host_check as mhc
    return mhc, mhc.build(str(tmp_path_factory.mktemp("mchg")))


def _lam_max_gc(theta, g, c, f):
    """Largest eigenvalue of the pencil with coefficients (g, c, f), symmetrised as marginal_oracle.lam_max does."""
    _, _, _, f_u, _, diag, sup = bo.discretise(theta, g, c, f)
    fi = f_u[1:-1]
    m = len(diag)
    return float(eigvalsh_tridiagonal(diag, sup * np.sqrt(fi[:-1] / fi[1:]), select="i", select_range=(m - 1, m - 1))[0])


def kappa_star_gc(theta, g, c1, c2, f, k0, rel=5e-2):
    """Oracle kappa* of the pencil with given g and c(kappa) = kappa c1 + kappa^2 c2 (f does not move the crossing), bracketed
    in k0 (1 -+ rel)."""
    lam = lambda k: _lam_max_gc(theta, g, k * c1 + k * k * c2, f)
    return brentq(lam, k0 * (1 - rel), k0 * (1 + rel), xtol=1e-15 * k0, rtol=8.9e-16, maxiter=200)


def _split(base, dP, th0):
    """g, c1, c2, f of one line: c(kappa) = kappa c1 + kappa^2 c2 (marginal_oracle.coefficients)."""
    b = base
    gd = b[GDS2] + 2 * th0 * b[GDS21] + th0 ** 2 * b[GDS22]
    g, c1, f = bo.gcf(dP, b[BMAG], b[GRADPAR], b[GBDRIFT] + th0 * b[CVDRIFT0], gd)
    c2 = bo.gcf(dP, b[BMAG], b[GRADPAR], b[CVDRIFT] - b[GBDRIFT], gd)[1]
    return g, c1, c2, f


def richardson(fun, eps=1e-3):
    """d/de fun(e) at 0: central differences at eps and eps / 2, Richardson-extrapolated.  kappa* of the oracle is accurate to
    ~1e-11 relative (eps |K| / (kappa dlam/dkappa)), so the steps stay large and the O(eps^2) error is extrapolated away."""
    d1 = (fun(eps) - fun(-eps)) / (2 * eps)
    d2 = (fun(eps / 2) - fun(-eps / 2)) / eps
    return (4 * d2 - d1) / 3


def _smooth(rng, theta, n):
    """n smooth random profiles on theta, O(1)."""
    L = theta[-1] - theta[0]
    out = np.zeros((n, theta.size))
    for k in range(1, 4):
        out += rng.standard_normal((n, 1)) * np.cos(np.pi * k * (theta - theta[0]) / L + rng.uniform(0, 2 * np.pi, (n, 1))) / k
    return out + rng.standard_normal((n, 1))


def _solve(harness, D):
    mhc, lib = harness
    base, dP = mhc.fixture_lines(D)
    theta = D["theta"]
    h = theta[1] - theta[0]
    nl, nt = base.shape[0], len(THETA0)
    R = mhc.solve(lib, base, dP, np.tile(THETA0, nl), h, nth0=nt, want_X=True)
    assert np.all((R["info"] >> 16) == 0)
    return base, dP, theta, h, R


@pytest.mark.parametrize("name", FIXTURES)
def test_alpha_tangent_is_directional_derivative(harness, golden, name):
    """-qa / qk along random smooth (dbase, ddPdrho) against the oracle's central difference of kappa*(base -+ eps dbase,
    dPdrho -+ eps ddPdrho) (Richardson), on every line of the fixture."""
    mhc, lib = harness
    base, dP, theta, h, R = _solve(harness, golden(name))
    nl, nt = base.shape[0], len(THETA0)
    rng = np.random.default_rng(11)
    dbase = np.stack([base[l] * _smooth(rng, theta, 8) for l in range(nl)])
    ddP = dP * rng.standard_normal(nl)
    got = mhc.tangent(lib, base, dbase, dP, ddP, np.tile(THETA0, nl), h, R["kappa"], R["X"], nth0=nt)
    worst = 0.0
    for line in range(nl):
        for t, th0 in enumerate(THETA0):
            s = line * nt + t
            k = R["kappa"][s]
            eps = 1e-3 * k / max(abs(got[s]), k)              # kappa* moves by ~1e-3 of itself
            fd = richardson(lambda e: mo.kappa_star(base[line] + e * dbase[line], dP[line] + e * ddP[line], theta, th0), eps)
            err = abs(got[s] - fd) / max(abs(fd), 1e-3 * k)
            worst = max(worst, err)
            assert err <= 1e-6, (line, t, got[s], fd)
    print(f"{name}: worst relative error of d kappa* / d alpha {worst:.1e}")


@pytest.mark.parametrize("name", FIXTURES)
def test_sensitivities_against_perturbed_coefficients(harness, golden, name):
    """sum_j (dk/dg_j dg_j + dk/dc_j dc_j) along random smooth (dg, dc) against the oracle's kappa* of the pencil with
    perturbed coefficients; dc is a change of c at kappa*, i.e. of c1 by dc / kappa*."""
    mhc, lib = harness
    base, dP, theta, h, R = _solve(harness, golden(name))
    nl, nt = base.shape[0], len(THETA0)
    th0 = np.tile(THETA0, nl)
    dk_dg, dk_dc = mhc.sensitivities(lib, base, dP, th0, h, R["kappa"], R["X"], nth0=nt)
    assert np.all(dk_dc[:, 0] == 0.0) and np.all(dk_dc[:, -1] == 0.0) and np.all(dk_dg >= 0.0) and np.all(dk_dc <= 0.0)
    rng = np.random.default_rng(5)
    for line in range(nl):
        for t in range(nt):
            s = line * nt + t
            k = R["kappa"][s]
            g, c1, c2, f = _split(base[line], dP[line], THETA0[t])
            dg = g * _smooth(rng, theta, 1)[0]
            dc = np.abs(k * c1 + k * k * c2).max() * _smooth(rng, theta, 1)[0]
            got = float(dk_dg[s] @ dg + dk_dc[s] @ dc)
            eps = 1e-3 * k / max(abs(got), k)
            want = richardson(lambda e: kappa_star_gc(theta, g + e * dg, c1 + e * dc / k, c2, f, k), eps)
            assert abs(got - want) <= 1e-6 * max(abs(want), 1e-3 * k), (line, t, got, want)


@pytest.mark.parametrize("name", FIXTURES)
def test_scale_identity(harness, golden, name):
    """sum_j g_j dk/dg_j + sum_j c_j dk/dc_j = -x^T K(kappa*) x / qk, which vanishes at the null vector."""
    mhc, lib = harness
    base, dP, theta, h, R = _solve(harness, golden(name))
    nl, nt = base.shape[0], len(THETA0)
    dk_dg, dk_dc = mhc.sensitivities(lib, base, dP, np.tile(THETA0, nl), h, R["kappa"], R["X"], nth0=nt)
    for line in range(nl):
        for t in range(nt):
            s = line * nt + t
            g, c, _ = mo.coefficients(base[line], dP[line], THETA0[t], R["kappa"][s])
            terms = np.concatenate([g * dk_dg[s], c * dk_dc[s]])
            assert abs(terms.sum()) <= 1e-10 * np.abs(terms).sum(), (line, t, terms.sum(), np.abs(terms).sum())


def test_theta0_tangent_reproduces_dkappa_dtheta0(harness, golden):
    """The tangent form along the theta0-direction of the records (d gds2 = 2 gds21 + 2 theta0 gds22, d cvdrift = cvdrift0 at
    fixed theta0 is the theta0 shift) gives the lane code's own d kappa* / d theta0: both forms are the same quadratic form."""
    mhc, lib = harness
    base, dP, theta, h, R = _solve(harness, golden("synthetic_ncsx"))
    nl, nt = base.shape[0], len(THETA0)
    for t, th0 in enumerate(THETA0):
        db = np.zeros_like(base)
        db[:, GDS2] = 2 * base[:, GDS21] + 2 * th0 * base[:, GDS22]
        db[:, CVDRIFT] = base[:, CVDRIFT0]
        db[:, GBDRIFT] = base[:, CVDRIFT0]
        sel = np.arange(nl) * nt + t
        got = mhc.tangent(lib, base, db, dP, np.zeros(nl), np.full(nl, th0), h, R["kappa"][sel], R["X"][sel])
        want = R["dkappa_dtheta0"][sel]
        np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-12 * np.abs(R["kappa"][sel]).max())
