"""TEST INFRASTRUCTURE ONLY -- CPU reference of the critical pressure-gradient factor kappa* (marginal stability).

kappa* of a field line at theta0 is the smallest factor of p' (at fixed geometry) at which the discrete ballooning pencil of
``ballooning_oracle.discretise`` has an eigenvalue above 0.  Scaling p' by kappa is, on the base arrays,
``cvdrift -> gbdrift + kappa (cvdrift - gbdrift)`` and ``dPdrho -> kappa dPdrho`` (K1 puts p' nowhere else).  Here the pencil is
symmetrised exactly as ``ballooning_oracle.gamma_ball_full(method="lambda_max")`` does, its top eigenvalue is taken with
LAPACK (``eigvalsh_tridiagonal``) and the zero crossing in kappa with ``brentq``; the derivatives are central differences.
"""
from __future__ import annotations

import numpy as np
from scipy.linalg import eigvalsh_tridiagonal
from scipy.optimize import brentq

from . import ballooning_oracle as bo

# rows of a base array (8, N): IBS_BASE_* order
BMAG, GRADPAR, CVDRIFT, CVDRIFT0, GDS2, GDS21, GDS22, GBDRIFT = range(8)


def coefficients(base, dPdrho, theta0, kappa):
    """g, c, f of one field line with p' scaled by ``kappa`` (``ball_scan.py:267-268`` + ``utils.py:1560-1562``)."""
    b = np.asarray(base, dtype=float)
    cv = b[GBDRIFT] + kappa * (b[CVDRIFT] - b[GBDRIFT]) + theta0 * b[CVDRIFT0]
    gd = b[GDS2] + 2 * theta0 * b[GDS21] + theta0 ** 2 * b[GDS22]
    return bo.gcf(kappa * dPdrho, b[BMAG], b[GRADPAR], cv, gd)


def lam_max(base, dPdrho, theta, theta0, kappa):
    """Largest eigenvalue of the discrete pencil (the matrix eigenvalue, not the Simpson quotient)."""
    g, c, f = coefficients(base, dPdrho, theta0, kappa)
    _, _, _, f_u, _, diag, sup = bo.discretise(theta, g, c, f)
    fi = f_u[1:-1]
    e = sup * np.sqrt(fi[:-1] / fi[1:])
    m = len(diag)
    return float(eigvalsh_tridiagonal(diag, e, select="i", select_range=(m - 1, m - 1))[0])


def kappa_star(base, dPdrho, theta, theta0, kappa_max=1e3):
    """kappa* by bracketing (doubling / halving from 1) and ``brentq`` on lam_max(kappa); ``inf`` without a crossing up to
    ``kappa_max``."""
    if dPdrho == 0.0:
        return np.inf
    f = lambda k: lam_max(base, dPdrho, theta, theta0, k)
    lo, hi = 1.0, 1.0
    if f(1.0) > 0.0:
        while f(lo) > 0.0:
            lo *= 0.5
        hi = 2 * lo
    else:
        while f(hi) <= 0.0:
            if hi >= kappa_max:
                return np.inf
            lo, hi = hi, min(2 * hi, kappa_max)
    return brentq(f, lo, hi, xtol=1e-15 * hi, rtol=8.9e-16, maxiter=200)


def dlam_dkappa(base, dPdrho, theta, theta0, kappa, rel=1e-5):
    d = rel * kappa
    return (lam_max(base, dPdrho, theta, theta0, kappa + d) - lam_max(base, dPdrho, theta, theta0, kappa - d)) / (2 * d)


def dkappa_dtheta0(base, dPdrho, theta, theta0, d=1e-5):
    return (kappa_star(base, dPdrho, theta, theta0 + d) - kappa_star(base, dPdrho, theta, theta0 - d)) / (2 * d)
