"""CPU: pin the oracle (oracle/ballooning_oracle.py) against the golden fixtures that were generated
from the UNMODIFIED reference (tests/golden/make_golden.py), and -- when /root/reference is present
(build container only) -- against the reference itself, live."""
import os

import numpy as np
import pytest

from helpers import fixture_gcf, sign_normalise, tables_from_fixture
from oracle import ballooning_oracle as bo
from oracle import ref_shim

FIXTURES = ["ncsx_wout_op", "synthetic_ncsx", "synthetic_d3d", "synthetic_hberg"]


@pytest.mark.parametrize("name", FIXTURES)
def test_fieldlines_match_reference_outputs(golden, name):
    """a1-a4: vmec_fieldlines restatement (utils.py:161-864) vs the reference's own arrays."""
    D = golden(name)
    tab = tables_from_fixture(D).select([0])           # one surface keeps the CPU suite fast
    fl = bo.fieldlines(tab, D["alphas"], D["theta"])
    np.testing.assert_allclose(fl.theta_vmec[0], D["theta_vmec"][0], rtol=0, atol=2e-12)
    for k in bo.HOT_FIELDS:
        ref = D["geo_" + k][0]
        scale = np.max(np.abs(ref), axis=-1, keepdims=True)
        assert np.max(np.abs(getattr(fl, k)[0] - ref) / scale) < 5e-12, k
    for ja in range(len(D["alphas"])):
        np.testing.assert_allclose(bo.dpdrho_of(fl, 0, ja), D["dPdrho"][0, ja], rtol=1e-11)


@pytest.mark.parametrize("name", FIXTURES)
def test_gamma_ball_full_matches_reference_outputs(golden, name):
    """a5-a8: the oracle's ARPACK route (tol=0) and its LAPACK cross-check vs the converged reference."""
    D = golden(name)
    theta = D["theta"]
    vg = bo.default_vguess(theta)
    i, j = 0, 0
    for k, th0 in enumerate(D["theta0s"][:2]):
        cv = D["geo_cvdrift"][i, j] + th0 * D["geo_cvdrift0"][i, j]
        gd = D["geo_gds2"][i, j] + 2 * th0 * D["geo_gds21"][i, j] + th0 ** 2 * D["geo_gds22"][i, j]
        args = (D["dPdrho"][i, j], theta, D["geo_bmag"][i, j], D["geo_gradpar_theta_pest"][i, j], cv, gd)
        lam_t, X_t, dX_t, g, c, f = bo.gamma_ball_full(*args, method="lambda_max")
        np.testing.assert_allclose(lam_t, D["lam_conv"][i, j, k], rtol=1e-10)
        np.testing.assert_allclose(sign_normalise(X_t), sign_normalise(D["X_conv"][i, j, k]), rtol=0, atol=1e-8)
        g2, c2, f2 = fixture_gcf(D, i, j, k)
        assert np.array_equal(g, g2) and np.array_equal(c, c2) and np.array_equal(f, f2)
        if k == 0:      # the dense ARPACK route is O(N^3): once per fixture
            lam_a, X_a, dX_a, *_ = bo.gamma_ball_full(*args, vg, 1.0, tol=0.0, method="arpack")
            np.testing.assert_allclose(lam_a, D["lam_conv"][i, j, k], rtol=1e-10)
            np.testing.assert_allclose(sign_normalise(X_a), sign_normalise(D["X_conv"][i, j, k]), rtol=0, atol=1e-8)
            np.testing.assert_allclose(sign_normalise(dX_a), sign_normalise(D["dX_conv"][i, j, k]) *
                                       np.sign(np.dot(sign_normalise(dX_a), sign_normalise(D["dX_conv"][i, j, k]))),
                                       rtol=0, atol=1e-7)


def test_s_alpha_known_answers(golden):
    """gamma_ball_full on the analytic s-alpha coefficients: converged reference values + the published
    stable/unstable labels of the reference's figure (bishop_ball_s-alpha.py:297-299)."""
    G = golden("s_alpha")
    theta = G["theta_512"]
    from ideal_ballooning_solver_b200 import synthetic
    for k, (sh, al, t0) in enumerate(G["cases"]):
        g, c, f = synthetic.s_alpha_coefficients(sh, al, t0, theta)
        one = np.ones_like(theta)
        lam, X, *_ = bo.gamma_ball_full(-al, theta, one, one, c / al, g, method="lambda_max")
        np.testing.assert_allclose(lam, G["lam_conv_512"][k], rtol=1e-10)
    lab = {(0.8, 0.8): True, (1.2, 0.2): False, (0.05, 1.0): False}       # (shat, alpha) -> unstable?
    for k, (sh, al, t0) in enumerate(G["cases"]):
        if t0 == 0.0 and (sh, al) in lab:
            assert (G["lam_conv_1024"][k] > 0) == lab[(sh, al)]


def test_check_ball_restatement(golden):
    """The Newcomb shooting test of the reference's s-alpha script (check_ball / check_ball_long)."""
    G = golden("s_alpha")
    for key, span, n in (("check_ball", 61, 1601), ("check_ball_long", 20, 401)):
        got = np.array([[bo.check_ball(sh, al, t0, span, n) for t0 in G["cb_theta0"]] for sh, al in G["cb_points"]])
        assert np.array_equal(got, G[key]), key


@pytest.mark.parametrize("name", ["synthetic_d3d", "synthetic_ncsx"])
def test_obj_w_grad_matches_reference_outputs(golden, name):
    """a9: adjoint gradient restatement (utils.py:1632-1728)."""
    D = golden(name)
    theta = D["theta"]
    si, al, th0, val, ga, gt = D["grad_points"][0]
    tab = tables_from_fixture(D).select([int(si)])
    v, grad = bo.obj_w_grad((al, th0), lambda alphas: bo.fieldlines(tab, alphas, theta), theta,
                            bo.default_vguess(theta), 1.0, method="lambda_max")
    np.testing.assert_allclose(v, val, rtol=1e-10)
    np.testing.assert_allclose(grad, [ga, gt], rtol=0, atol=1e-8)


def test_argmax_guards():
    """ball_scan.py:279-295."""
    g = np.zeros((4, 5))
    assert bo.argmax_with_guards(g) == (-1, -1, 0.05)
    g[2, 3] = g[1, 4] = 0.25
    ia, it, s0 = bo.argmax_with_guards(g)
    assert (ia, it) == (1, 4) and s0 == 1.3 * 0.25 + 0.05
    g = -np.ones((3, 3)); g[2, 1] = -0.5
    assert bo.argmax_with_guards(g)[:2] == (2, 1)


def test_scan_theta_grid():
    assert len(bo.scan_theta_grid(80, 0)) == 641 and len(bo.scan_theta_grid(11, 11)) == 969   # ball_scan.py:201-208


LIVE_SMALL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "live_small.npz")


def _live_small_sources():
    """The reference's outputs for the small case of ``live_small_fixture`` (tests/golden/make_golden.py): as stored in
    tests/golden/live_small.npz, and computed live when the unmodified reference is importable."""
    if os.path.isfile(LIVE_SMALL):
        D = np.load(LIVE_SMALL)
        yield "stored", {k: D[k] for k in D.files}
    if ref_shim.reference_available():
        import importlib.util
        spec = importlib.util.spec_from_file_location("make_golden", os.path.join(os.path.dirname(LIVE_SMALL), "make_golden.py"))
        make_golden = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(make_golden)
        yield "live", make_golden.live_small(make_golden.u)


@pytest.mark.skipif(not (os.path.isfile(LIVE_SMALL) or ref_shim.reference_available()),
                    reason="neither tests/golden/live_small.npz nor the unmodified reference (IBS_REFERENCE_ROOT) is present")
def test_live_reference_small():
    """The unmodified reference (its stored outputs, and live through oracle/ref_shim.py when present) vs the restatement on
    a small case: its own splines and field line on a synthetic D3D-like equilibrium, then gamma_ball_full at theta0 = 0.3."""
    from ideal_ballooning_solver_b200 import synthetic, tables
    theta = np.linspace(-2 * np.pi, 2 * np.pi, 129)
    tab = tables.RadialSplines(synthetic.make_equilibrium("d3d", seed=5)).evaluate([0.6])
    fl = bo.fieldlines(tab, np.array([0.4]), theta)
    dP = bo.dpdrho_of(fl)
    cv, gd = bo.theta0_shift(fl, 0.3)
    got = bo.gamma_ball_full(dP, theta, fl.bmag[0][0], fl.gradpar_theta_pest[0][0], cv, gd, method="lambda_max")
    for source, ref in _live_small_sources():
        for k in bo.HOT_FIELDS:
            r = ref["geo_" + k]
            assert np.max(np.abs(getattr(fl, k)[0][0] - r)) / np.max(np.abs(r)) < 1e-9, (source, k)
        np.testing.assert_allclose(got[0], ref["lam_conv"], rtol=1e-10, err_msg=source)
        np.testing.assert_allclose(sign_normalise(got[1]), sign_normalise(ref["X_conv"]), rtol=0, atol=1e-8, err_msg=source)


def _derm_cases(G):
    for key in G.files:
        if not key.startswith("derm"):
            continue
        fn, dim, ch, par = key.split("_")
        a = G["a1"] if dim == "1d" else G["a2"]
        b = None if fn == "derm" else (G["b1"] if dim == "1d" else (G["b2l"] if ch == "l" else G["b2r"]))
        yield key, fn, a, b, ch, par


def test_derm_dermv_restatement_matches_reference_golden(golden):
    """f4 (part): the curvature penalty's finite-difference helpers, against vectors produced by the unmodified reference
    (tests/golden/make_golden_derm.py) -- bit-exact, shapes included."""
    G = golden("derm")
    n = 0
    for key, fn, a, b, ch, par in _derm_cases(G):
        r = bo.derm(a, ch, par) if fn == "derm" else bo.dermv(a, b, ch, par)
        assert r.shape == G[key].shape and np.array_equal(r, G[key]), key
        n += 1
    assert n == 14


@pytest.mark.parametrize("case", ["fl_theta", "fl_phi", "axisym"])
def test_full_struct_restatement_matches_reference_fixture(golden, case):
    """f4: the oracle's restatement of the whole vmec_fieldlines / vmec_fieldlines_axisym Struct against the fixture the
    unmodified reference produced (tests/golden/make_golden_full.py)."""
    from ideal_ballooning_solver_b200.tables import SurfaceTables
    D = golden("full_struct")
    g = lambda k: np.array(D[f"{case}__in_{k}"])
    st = SurfaceTables(g("tab_mn"), g("tab_nyq"), g("scal"), g("xm"), g("xn"), g("xm_nyq"), g("xn_nyq"), float(g("phiedge")),
                       float(g("Aminor_p")), int(g("nfp")), bsupumnc=g("bsupumnc"), raxis_cc=g("raxis_cc"))
    kw = dict(phi_center=float(g("phi_center")))
    if case == "fl_phi":
        kw["phi1d"] = g("phi1d")
    else:
        kw["theta1d"] = g("theta1d")
    o = bo.fieldlines_full(st, g("alpha"), axisym=(case == "axisym"), **kw)
    n = 0
    for key in D.files:
        if not key.startswith(case + "__") or key.startswith(case + "__in_"):
            continue
        name = key[len(case) + 2:]
        if not hasattr(o, name):
            continue                    # per-surface scalars and bookkeeping entries are formed by the facade, not here
        want, got = np.asarray(D[key]), np.asarray(getattr(o, name), dtype=float)
        assert got.shape == want.shape, name
        scale = max(float(np.max(np.abs(want))), 1e-300)
        assert float(np.max(np.abs(got - want))) / scale < (2e-9 if name.endswith("_alternate") else 1e-11), (case, name)
        n += 1
    assert n >= (85 if case == "axisym" else 75)
