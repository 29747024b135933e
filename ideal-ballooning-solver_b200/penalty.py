"""Consumer side of the scan (SURVEY.md section 8 row f3, first half): the ballooning term of the outer objective and
its forward-difference Jacobian, exactly as the reference's optimiser forms them.

``sims_runner_NCSX.py:313``:  ``f0 = f0 + prefac[-1] * sum(max(gamma_ball - gamma_ball_thresh, 0))``, returned as ``sqrt(f0)``;
``sims_runner_NCSX.py:254-261``: ``df0[i] = (f0_i - f0_0) / step_i * 0.5 / sqrt(f0_0)``.
Second half of f3: ``hf_jacobian`` forms the same Jacobian from ONE scan of the base equilibrium plus the first-order
change of every surface's maximum growth rate under each perturbed equilibrium instead of ``ndofs + 1`` full scans.  That
change comes either from ``scan.table_gradient(..., scalars=True).predict(tables0, tables_pert)`` -- reverse mode through
K1 (``ibs_geometry_adjoint_scal``): the gradient with respect to every Fourier table coefficient, the surface scalars (iota,
iota', p', shat, s), phiedge and Aminor_p once, then one dot product per degree of freedom (``scalars=False`` counts the
Fourier tables only: enough for DOFs that move neither iota, the pressure nor phiedge) -- or from
``scan.hellmann_feynman_gamma`` (K1 on the arg-max field lines of each perturbed table set + one K4 contraction, no
eigen-solve), its finite-perturbation form.
The perturbed equilibria themselves (VMEC runs) stay outside this package.
"""
from __future__ import annotations

import numpy as np

GAMMA_BALL_THRESH = {"D3D": -0.0002, "NCSX": -0.0002, "HBERG": -0.0003}   # sims_runner_{D3D:57,NCSX:56,HBERG:55}.py
PREFAC_BALL = 50.0                                                          # sims_runner_NCSX.py:57 (prefac[-1])


def ballooning_penalty(gamma_ball, thresh: float = GAMMA_BALL_THRESH["NCSX"], prefac: float = PREFAC_BALL) -> float:
    """``prefac * sum(max(gamma - thresh, 0))`` over the surfaces of one equilibrium."""
    g = np.asarray(gamma_ball, dtype=np.float64)
    return float(prefac * np.sum(np.maximum(g - thresh, 0.0)))


def objective(f0_other: float, gamma_ball, thresh: float = GAMMA_BALL_THRESH["NCSX"], prefac: float = PREFAC_BALL,
              converged: bool = True) -> float:
    """``fobj`` of ``sims_runner_NCSX.py:279-318``: ``sqrt(other penalties + ballooning penalty)``; 9999 if VMEC failed."""
    if not converged:
        return float(np.sqrt(9999.0))
    return float(np.sqrt(f0_other + ballooning_penalty(gamma_ball, thresh, prefac)))


def fd_jacobian(f0_other, gamma_ball_all, step_arr, thresh: float = GAMMA_BALL_THRESH["NCSX"], prefac: float = PREFAC_BALL):
    """``dfobj`` of ``sims_runner_NCSX.py:245-262``: row 0 of the Jacobian of ``sqrt(f0)`` by forward differences over the
    ``ndofs + 1`` perturbed equilibria.  ``f0_other[i]``, ``gamma_ball_all[i]`` belong to equilibrium ``i`` (0 = base)."""
    f0_other = np.asarray(f0_other, dtype=np.float64)
    n = len(f0_other)
    f = np.array([f0_other[i] + ballooning_penalty(gamma_ball_all[i], thresh, prefac) for i in range(n)])
    df = np.zeros((1, n))
    for i in range(1, n):
        df[0, i] = (f[i] - f[0]) / step_arr[i] * 0.5 * 1 / np.sqrt(f[0])
    return f, df


def hf_jacobian(f0_other, gamma_base, dgamma, step_arr, thresh: float = GAMMA_BALL_THRESH["NCSX"], prefac: float = PREFAC_BALL):
    """As ``fd_jacobian``, with the growth rates of the perturbed equilibria predicted to first order:
    ``gamma_i = gamma_base + dgamma[i - 1]`` (``scan.TableGradient.predict`` or ``scan.hellmann_feynman_gamma``).  ``f0_other`` has ``ndofs + 1`` entries
    (0 = base), ``dgamma`` is ``(ndofs, ns)``."""
    gamma_base = np.asarray(gamma_base, dtype=np.float64)
    dgamma = np.asarray(dgamma, dtype=np.float64).reshape(-1, gamma_base.size)
    gam_all = [gamma_base] + [gamma_base + d for d in dgamma]
    return fd_jacobian(f0_other, gam_all, step_arr, thresh, prefac)
