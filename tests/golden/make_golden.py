#!/usr/bin/env python
"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Run in the build container (needs ``/root/reference``):

    python tests/golden/make_golden.py

It imports ``/root/reference/utils.py`` through ``oracle/ref_shim.py`` (two shims, see there)
and stores inputs + reference outputs as ``.npz`` files.  The fixtures travel to the GPU box,
the reference does not.  "conv" = ARPACK ``tol=0`` (converged reference, the parity target);
"ship" = the reference's shipped ``tol=5e-7``.
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
warnings.simplefilter("ignore")

from oracle import ref_shim  # noqa: E402
from ideal_ballooning_solver_b200 import synthetic  # noqa: E402
from ideal_ballooning_solver_b200.tables import TAB_MN_ROWS, TAB_NYQ_ROWS  # noqa: E402

u = ref_shim.load_reference_utils()
HOT = ["bmag", "gradpar_theta_pest", "cvdrift", "cvdrift0", "gds2", "gds21", "gds22", "gbdrift"]
SUMS = ["R", "d_R_d_s", "d_R_d_theta_vmec", "d_R_d_phi", "d_Z_d_s", "d_Z_d_theta_vmec", "d_Z_d_phi",
        "d_lambda_d_s", "d_lambda_d_theta_vmec", "d_lambda_d_phi", "sqrt_g_vmec", "modB", "d_B_d_s",
        "d_B_d_theta_vmec", "d_B_d_phi", "B_sup_phi", "B_sub_s", "B_sub_theta_vmec", "B_sub_phi"]


def vguess_of(theta, theta_fac=4):
    return (1 - np.tanh(theta[1:-1] / np.pi) ** 2) * np.cos(theta[1:-1] / (2 * theta_fac))


def ref_tables(vs, s):
    """Per-surface tables evaluated with the reference's own FITPACK spline objects
    (utils.py:311-357), in the engine's (ns, row, mn) layout."""
    s = np.atleast_1d(np.asarray(s, float))
    tab_mn = np.stack([np.stack([spl(s) for spl in getattr(vs, name)], axis=1) for name in TAB_MN_ROWS], axis=1)
    tab_nyq = np.stack([np.stack([spl(s) for spl in getattr(vs, name)], axis=1) for name in TAB_NYQ_ROWS], axis=1)
    iota, diota = vs.iota(s), vs.d_iota_d_s(s)
    scal = np.zeros((s.size, 8))
    scal[:, 0], scal[:, 1], scal[:, 2] = s, iota, diota
    scal[:, 3] = vs.d_pressure_d_s(s)
    scal[:, 4] = (-2 * s / iota) * diota
    scal[:, 5] = vs.pressure(s)
    return tab_mn, tab_nyq, scal


def solve_both(dP, theta, fl, ja, th0, vg, sigma):
    cv = fl.cvdrift[0][ja] + th0 * fl.cvdrift0[0][ja]
    gd = fl.gds2[0][ja] + 2 * th0 * fl.gds21[0][ja] + th0 ** 2 * fl.gds22[0][ja]
    args = (dP, theta, fl.bmag[0][ja], fl.gradpar_theta_pest[0][ja], cv, gd, vg, sigma)
    ship = u.gamma_ball_full(*args)
    with ref_shim.converged_arpack(u):
        conv = u.gamma_ball_full(*args)
    return ship, conv


def equilibrium_fixture(name, wout, surfaces, alphas, theta0s, theta, grad_points, scan=None):
    vs = u.vmec_splines(ref_shim.FakeVmec(wout))
    out = dict(theta=theta, surfaces=np.array(surfaces), alphas=np.array(alphas), theta0s=np.array(theta0s),
               xm=vs.xm, xn=vs.xn, xm_nyq=vs.xm_nyq, xn_nyq=vs.xn_nyq, phiedge=vs.phiedge,
               Aminor_p=vs.Aminor_p, nfp=vs.nfp)
    out["tab_mn"], out["tab_nyq"], out["scal"] = ref_tables(vs, surfaces)
    vg = vguess_of(theta)
    ns, na, nt = len(surfaces), len(alphas), len(theta0s)
    nl = len(theta)
    for k in HOT:
        out["geo_" + k] = np.zeros((ns, na, nl))
    out["theta_vmec"] = np.zeros((ns, na, nl))
    for k in SUMS:
        out["sum_" + k] = np.zeros((ns, nl))          # first alpha only (keeps the file small)
    out["dPdrho"] = np.zeros((ns, na))
    for tag in ("ship", "conv"):
        out[f"lam_{tag}"] = np.zeros((ns, na, nt))
    out["X_conv"] = np.zeros((ns, na, nt, nl))
    out["dX_conv"] = np.zeros((ns, na, nt, nl))
    for i, s in enumerate(surfaces):
        fl = u.vmec_fieldlines(vs, s, np.array(alphas), theta1d=theta)
        for k in HOT:
            out["geo_" + k][i] = getattr(fl, k)[0]
        out["theta_vmec"][i] = fl.theta_vmec[0]
        for k in SUMS:
            out["sum_" + k][i] = getattr(fl, k)[0][0]
        for j in range(na):
            dP = -1.0 * 0.5 * np.mean((fl.cvdrift[0][j] - fl.gbdrift[0][j]) * fl.bmag[0][j] ** 2)
            out["dPdrho"][i, j] = dP
            for k, th0 in enumerate(theta0s):
                ship, conv = solve_both(dP, theta, fl, j, th0, vg, 1.0)
                out["lam_ship"][i, j, k] = ship[0]
                out["lam_conv"][i, j, k] = conv[0]
                out["X_conv"][i, j, k] = conv[1]
                out["dX_conv"][i, j, k] = conv[2]
    # obj_w_grad (utils.py:1632) at a few points, converged
    gp = []
    for (si, al, th0) in grad_points:
        with ref_shim.converged_arpack(u):
            val, grad = u.obj_w_grad((al, th0), vs, surfaces[si], theta, vg, 1.0)
        gp.append([si, al, th0, val, grad[0], grad[1]])
    out["grad_points"] = np.array(gp)
    if scan is not None:
        # coarse scan with the warm-start chain of ball_scan.py:248-274 (converged)
        si, a_scan, t_scan = scan
        vguess = vg.copy()
        gam = np.zeros((len(a_scan), len(t_scan)))
        with ref_shim.converged_arpack(u):
            for i, al in enumerate(a_scan):
                fl = u.vmec_fieldlines(vs, surfaces[si], al, theta1d=theta)
                bm = fl.bmag[0][0]
                dP = -1.0 * 0.5 * np.mean((fl.cvdrift[0][0] - fl.gbdrift[0][0]) * bm ** 2)
                for j, th0 in enumerate(t_scan):
                    cv = fl.cvdrift[0][0] + th0 * fl.cvdrift0[0][0]
                    gd = fl.gds2[0][0] + 2 * th0 * fl.gds21[0][0] + th0 ** 2 * fl.gds22[0][0]
                    lam, X, *_ = u.gamma_ball_full(dP, theta, bm, fl.gradpar_theta_pest[0][0], cv, gd, vguess, 1.0)
                    vguess = X[1:-1]
                    gam[i, j] = lam
        out["scan_surface"], out["scan_alpha"], out["scan_theta0"], out["scan_gamma"] = si, a_scan, t_scan, gam
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "lam_conv range", out["lam_conv"].min(), out["lam_conv"].max(),
          "max |ship-conv|/|conv|", np.max(np.abs(out["lam_ship"] / out["lam_conv"] - 1)))


def s_alpha_fixture():
    """gamma_ball_full on the analytic s-alpha coefficients (SURVEY 8c): B = gradpar = 1,
    gds2 = 1+Lambda^2, cvdrift = cos + Lambda sin, dPdrho = -alpha."""
    cases = [(0.8, 0.8, 0.0), (1.0, 0.9, 0.0), (0.4, 0.4, 0.0), (1.2, 0.2, 0.0), (1.6, 0.6, 0.0),
             (0.05, 1.0, 0.0), (0.8, 0.8, 0.2), (0.3, 0.6, 0.1), (2.0, 1.2, 0.0), (0.6, 0.1, 0.1)]
    out = dict(cases=np.array(cases))
    for nth, span in ((1024, 10), (2048, 10), (512, 4)):
        theta = np.linspace(-span * np.pi, span * np.pi, nth + 1)
        vg = vguess_of(theta, theta_fac=span)
        lam_s, lam_c, Xs, dXs = [], [], [], []
        for shat, al, th0 in cases:
            g, c, f = synthetic.s_alpha_coefficients(shat, al, th0, theta)
            one = np.ones_like(theta)
            args = (-al, theta, one, one, c / al, g, vg, 2.0)
            lam_s.append(u.gamma_ball_full(*args)[0])
            with ref_shim.converged_arpack(u):
                r = u.gamma_ball_full(*args)
            lam_c.append(r[0]); Xs.append(r[1]); dXs.append(r[2])
        out[f"theta_{nth}"] = theta
        out[f"lam_ship_{nth}"], out[f"lam_conv_{nth}"] = np.array(lam_s), np.array(lam_c)
        out[f"X_conv_{nth}"], out[f"dX_conv_{nth}"] = np.array(Xs), np.array(dXs)
        print("s-alpha", nth, np.array(lam_c))
    # marginal-stability classification of the reference's own s-alpha test
    cb, cbl = ref_shim.load_s_alpha_checkers()
    pts = [(0.8, 0.8), (1.2, 0.2), (0.05, 1.0), (0.4, 0.4), (1.6, 0.6), (1.0, 0.9), (0.3, 0.6), (2.0, 1.2),
           (0.6, 0.1), (1.0, 0.5), (0.2, 0.3), (1.5, 1.1)]
    out["cb_points"] = np.array(pts)
    out["cb_theta0"] = np.array([0.0, 0.1, 0.2])
    out["check_ball"] = np.array([[cb(sh, al, t0) for t0 in out["cb_theta0"]] for sh, al in pts])
    out["check_ball_long"] = np.array([[cbl(sh, al, t0) for t0 in out["cb_theta0"]] for sh, al in pts])
    print("check_ball", out["check_ball"].T.tolist())
    np.savez_compressed(os.path.join(HERE, "s_alpha.npz"), **out)


def live_small(u):
    """The small case of tests/test_oracle.py::test_live_reference_small: the reference's own splines and field line on a
    synthetic D3D-like equilibrium (seed 5, s = 0.6, alpha = 0.4, 129 points on +-2 pi), and its converged gamma_ball_full at
    theta0 = 0.3 on the restatement's coefficients of that line (so that the eigensolvers see identical input)."""
    from oracle import ballooning_oracle as bo
    from ideal_ballooning_solver_b200 import tables
    wout = synthetic.make_equilibrium("d3d", seed=5)
    theta = np.linspace(-2 * np.pi, 2 * np.pi, 129)
    fl_ref = u.vmec_fieldlines(u.vmec_splines(ref_shim.FakeVmec(wout)), 0.6, np.array([0.4]), theta1d=theta)
    out = {"geo_" + k: getattr(fl_ref, k)[0][0] for k in bo.HOT_FIELDS}
    fl = bo.fieldlines(tables.RadialSplines(wout).evaluate([0.6]), np.array([0.4]), theta)
    cv, gd = bo.theta0_shift(fl, 0.3)
    with ref_shim.converged_arpack(u):
        out["lam_conv"], out["X_conv"], *_ = u.gamma_ball_full(bo.dpdrho_of(fl), theta, fl.bmag[0][0], fl.gradpar_theta_pest[0][0],
                                                               cv, gd, bo.default_vguess(theta), 1.0)
    return out


def live_small_fixture():
    out = live_small(u)
    np.savez_compressed(os.path.join(HERE, "live_small.npz"), **out)
    print("live_small lam_conv", out["lam_conv"])


if __name__ == "__main__":
    if sys.argv[1:] == ["live_small"]:
        live_small_fixture()
        sys.exit(0)
    live_small_fixture()
    s_alpha_fixture()
    # the only real equilibrium shipped with the reference
    wout = ref_shim.wout_from_netcdf(os.path.join(ref_shim.REFERENCE_ROOT, "tests", "comparn_w_COBRAVMEC",
                                                  "wout_NCSX_op.nc"))
    th969 = np.linspace(-4 * np.pi, 4 * np.pi, 969)
    equilibrium_fixture("ncsx_wout_op", wout, [0.5, 0.7, 0.9, 0.95], [0.0, 0.3, 1.0, 2.0], [0.0, 0.5, 1.0], th969,
                        grad_points=[(1, 0.3, 0.1), (0, 1.0, 0.5), (2, 2.0, 0.0)],
                        scan=(1, np.linspace(0, np.pi, 4), np.linspace(0, 0.5 * np.pi, 5)))
    # synthetic equilibria at the three device mode counts
    equilibrium_fixture("synthetic_ncsx", synthetic.make_equilibrium("ncsx"), [0.5, 0.7, 0.9], [0.0, 1.3], [0.0, 0.8],
                        np.linspace(-4 * np.pi, 4 * np.pi, 1025), grad_points=[(0, 1.3, 0.4), (1, 0.2, 0.0)],
                        scan=(0, np.linspace(0, np.pi, 3), np.linspace(0, 0.5 * np.pi, 4)))
    equilibrium_fixture("synthetic_d3d", synthetic.make_equilibrium("d3d"), [0.5, 0.8, 0.95], [0.0], [0.0, 0.7, 1.4],
                        np.linspace(-4 * np.pi, 4 * np.pi, 1025), grad_points=[(1, 0.0, 0.3)])
    equilibrium_fixture("synthetic_hberg", synthetic.make_equilibrium("hberg"), [0.6, 0.9], [0.5, 2.5], [0.0, 1.0],
                        np.linspace(-8 * np.pi, 8 * np.pi, 2049), grad_points=[(0, 0.5, 0.2)])
