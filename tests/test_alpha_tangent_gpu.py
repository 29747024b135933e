"""Exact alpha-derivative of the growth rate: the alpha-tangent of K1 (``ibs_geometry_tangent_batch``) and the ``obj_w_grad``
contraction that consumes it (``ibs_obj_w_grad_tangent_batch``), and ``scan.refine_maxima(..., alpha_derivative="exact")``.

Argument checks without a GPU; on the GPU: the value outputs equal ``geometry_batch``'s bit for bit on every kernel shape; the
tangent against Richardson-extrapolated central differences of the long-double field-line reference; the gradient against the
three-line finite-difference path (bit-identical value, theta0 part, eigenfunction and flags; the finite difference converges
to it at second order), against re-solved eigenvalues, and in the refinement of 64 surfaces."""

import numpy as np
import pytest

from helpers import tables_from_fixture
from geometry_ld import LD, fieldlines_ld
from test_geometry_shapes_gpu import SHAPES, Shape

FIXTURES = ["synthetic_d3d", "synthetic_ncsx", "synthetic_hberg", "ncsx_wout_op"]
NBASE = 8

# Each d base / d alpha row within TAN_RTOL of its maximum (d dPdrho / d alpha of the line's |dPdrho|).  Worst case measured on an
# NVIDIA B200 (1000 W power limit) over all shapes and fixtures: 1.2e-12 (the gradpar row of the 4097-point lines).
TAN_RTOL = 1e-11


def _fieldlines_ld_alpha(tab, alpha, theta, phi_center=0.0, cols=None):
    """``fieldlines_ld`` with alpha and phi = phi_center + (theta - alpha) / iota in long double, so that central differences
    in alpha with steps ~1e-5 are not limited by the float64 rounding of phi."""
    return fieldlines_ld(tab, np.asarray(alpha, dtype=LD), theta, phi_center, cols, phi_ld=True)


def richardson_alpha(tab, alpha, theta, phi_center, cols, h=2.0 ** -15):
    """d/d alpha of the reference's eight base arrays (and of the line mean that dPdrho takes when ``cols`` is the whole line):
    central differences at h and h / 2, Richardson-extrapolated, in long double."""
    from ideal_ballooning_solver_b200.engine import BASE_NAMES
    a = np.asarray(alpha, dtype=LD)

    def arrays(da):
        r = _fieldlines_ld_alpha(tab, a + LD(da), theta, phi_center, cols)
        b = np.stack([r[n] for n in BASE_NAMES], axis=2)
        dp = -0.5 * np.mean((r["cvdrift"] - r["gbdrift"]) * r["bmag"] ** 2, axis=-1)
        return b, dp

    def central(hh):
        (bp, dpp), (bm, dpm) = arrays(hh), arrays(-hh)
        return (bp - bm) / LD(2 * hh), (dpp - dpm) / LD(2 * hh)

    (b1, d1), (b2, d2) = central(h), central(h / 2)
    return ((4 * b2 - b1) / 3).astype(np.float64), ((4 * d2 - d1) / 3).astype(np.float64)


def _tables(st):
    from ideal_ballooning_solver_b200 import engine
    return engine.DeviceTables.from_host(st)


def _both(st, alpha, theta, phi_center=0.0):
    import torch
    from ideal_ballooning_solver_b200 import engine
    dt = _tables(st)
    a = torch.from_numpy(np.ascontiguousarray(alpha, dtype=np.float64)).cuda()
    t = torch.from_numpy(np.asarray(theta, dtype=np.float64)).cuda()
    g = engine.geometry_batch(dt, a, t, phi_center=phi_center, want_theta_vmec=True, want_info=True)
    gt = engine.geometry_tangent_batch(dt, a, t, phi_center=phi_center, want_theta_vmec=True, want_info=True)
    return g, gt


def _rate(st):
    """|d phi / d alpha| = 1 / |iota| of each surface, shaped (ns, 1, 1): turns a base array's size into the size of its
    alpha-derivative if it varied at the rate the field line moves."""
    return (1.0 / np.abs(np.asarray(st.scal)[:, 1]))[:, None, None]


def _row_err(got, want, base, rate):
    """max over rows (the last axis) of max |got - want| / max |got|.  A row whose reference derivative is zero to rounding
    (gds22 of axisymmetric tables: grad psi does not depend on alpha there) has no scale of its own; its tangent must be zero to
    the rounding of the Cartesian algebra, measured against max |base row| / |iota|.  Degeneracy is read from the reference."""
    deriv_scale = np.max(np.abs(base), axis=-1, keepdims=True) * rate
    zero = np.max(np.abs(want), axis=-1, keepdims=True) <= 1e-12 * deriv_scale
    scale = np.where(zero, deriv_scale, np.max(np.abs(got), axis=-1, keepdims=True))
    return float(np.max(np.abs(got - want) / scale))


def _ddp_err(got, want, dP, rate):
    """d dPdrho / d alpha against the reference, relative to |dPdrho| / |iota| per line: (cvdrift - gbdrift) bmag^2 is the same
    constant at every point of a line, so the derivative is zero to rounding."""
    return float(np.max(np.abs(got - want) / (np.abs(dP) * rate[:, :, 0])))


# ---------------------------------------------------------------------------------------------------------------------
# host-side argument checks (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
def test_argument_errors_without_gpu():
    """Both entry points reject what ibs_geometry_batch and ibs_obj_w_grad_batch reject, before any CUDA call, with a message;
    empty batches return 0."""
    from ideal_ballooning_solver_b200 import _lib, build
    build.build()
    lib = _lib.load()
    buf = np.zeros(64)
    p = buf.ctypes.data

    def geo(ns=2, nalpha=3, nl=9, ptr=p, dbase=p, base=p, phiedge=0.5, aminor_p=0.3, mnmax=3):
        return lib.ibs_geometry_tangent_batch(ptr, ptr, ptr, ptr, ptr, ptr, ptr, ns, mnmax, 4, phiedge, aminor_p, ptr, nalpha, 0, ptr,
                                              nl, 0.0, base, p, dbase, None, None, None, None)
    assert geo(ns=0) == 0 and geo(nalpha=0) == 0
    assert geo(ptr=None) == 1 and b"null" in lib.ibs_last_error()
    assert geo(dbase=None) == 1 and b"null" in lib.ibs_last_error()
    assert geo(base=None) == 1 and b"null" in lib.ibs_last_error()
    assert geo(ns=-1) == 1 and b"bad sizes" in lib.ibs_last_error()
    assert geo(nalpha=-2) == 1 and b"bad sizes" in lib.ibs_last_error()
    assert geo(nl=0) == 1 and b"bad sizes" in lib.ibs_last_error()
    assert geo(mnmax=0) == 1 and b"bad sizes" in lib.ibs_last_error()
    assert geo(aminor_p=0.0) == 1 and b"Aminor_p" in lib.ibs_last_error()
    assert geo(phiedge=0.0) == 1 and b"phiedge" in lib.ibs_last_error()

    def owg(npoint=4, N=65, h=0.1, base=p, dbase=p, ddp=p, val=p):
        return lib.ibs_obj_w_grad_tangent_batch(base, dbase, p, ddp, p, npoint, N, h, None, val, p, None, None, None, None)
    assert owg(npoint=0) == 0
    assert owg(npoint=-1) == 1 and b"bad sizes" in lib.ibs_last_error()
    assert owg(N=4) == 1 and b"bad sizes" in lib.ibs_last_error()
    assert owg(h=0.0) == 1 and b"bad sizes" in lib.ibs_last_error()
    assert owg(h=-0.1) == 1 and b"bad sizes" in lib.ibs_last_error()
    for kw in ("base", "dbase", "ddp", "val"):
        assert owg(**{kw: None}) == 1 and b"null" in lib.ibs_last_error(), kw


def test_refine_rejects_unknown_alpha_derivative_without_gpu():
    from ideal_ballooning_solver_b200 import scan
    with pytest.raises(ValueError, match="alpha_derivative"):
        scan.refine_maxima(None, [0.0], [0.0], np.linspace(-1, 1, 9), alpha_derivative="central")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: values bit-identical to geometry_batch; tangent against the extended-precision reference
# ---------------------------------------------------------------------------------------------------------------------
def _value_cases():
    cases = []
    for name, spec in SHAPES.items():
        cases.append((name, "default"))
        if spec["ntor"] == 0:
            cases.append((name, "fold-off"))
    for name in ("ntor5_nfp3", "ntor11_nfp3", "ntor16_nfp2"):
        cases.append((name, "geo3d"))
    return cases


@pytest.fixture(scope="module")
def shapes():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = Shape(name, SHAPES[name])
        return cache[name]
    return get


def _env(monkeypatch, mode):
    if mode == "fold-off":
        monkeypatch.setenv("IBS_GEO_FOLD", "0")
    if mode == "geo3d":
        monkeypatch.setenv("IBS_GEO3D", "1")


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _value_cases())
def test_values_bit_identical_to_geometry_batch(cuda_lib, shapes, monkeypatch, name, mode):
    """base, dPdrho, theta_vmec and info of the tangent entry point are geometry_batch's bits: every kernel shape, the fold on
    and off, IBS_GEO3D=1, alpha shared and per surface (the per_surface_alpha shapes)."""
    sh = shapes(name)
    _env(monkeypatch, mode)
    g, gt = _both(sh.st, sh.alpha, sh.theta, sh.phi_center)
    for a, b in ((g.base, gt.base), (g.dPdrho, gt.dPdrho), (g.theta_vmec, gt.theta_vmec), (g.info, gt.info)):
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy()), (name, mode)
    assert np.all(np.isfinite(gt.dbase.cpu().numpy())) and np.all(np.isfinite(gt.ddPdrho.cpu().numpy()))


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", _value_cases())
def test_tangent_matches_extended_precision_reference(cuda_lib, shapes, monkeypatch, name, mode):
    """Each d base / d alpha row within TAN_RTOL of its maximum against Richardson central differences of the long-double
    reference; d dPdrho / d alpha likewise where the reference covers the whole line."""
    sh = shapes(name)
    _env(monkeypatch, mode)
    _, gt = _both(sh.st, sh.alpha, sh.theta, sh.phi_center)
    db, ddp = richardson_alpha(sh.st, sh.alpha, sh.theta, sh.phi_center, sh.cols)
    got = gt.dbase.cpu().numpy()
    base = gt.base.cpu().numpy()
    errs = [_row_err(got[:, :, k, :][..., sh.cols], db[:, :, k, :], base[:, :, k, :], _rate(sh.st)) for k in range(NBASE)]
    print(name, mode, "dbase row errors", ["%.1e" % e for e in errs])
    assert max(errs) < TAN_RTOL, (name, mode, errs)
    if sh.cols.size == sh.theta.size:
        err = _ddp_err(gt.ddPdrho.cpu().numpy(), ddp, gt.dPdrho.cpu().numpy(), _rate(sh.st))
        print(name, mode, "ddPdrho error %.1e" % err)
        assert err < TAN_RTOL, (name, mode, err)


@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXTURES)
def test_tangent_matches_reference_on_fixtures(cuda_lib, golden, name):
    D = golden(name)
    st = tables_from_fixture(D)
    theta, alpha = D["theta"], D["alphas"]
    _, gt = _both(st, alpha, theta)
    db, ddp = richardson_alpha(st, alpha, theta, 0.0, np.arange(theta.size))
    got = gt.dbase.cpu().numpy()
    base = gt.base.cpu().numpy()
    errs = [_row_err(got[:, :, k, :], db[:, :, k, :], base[:, :, k, :], _rate(st)) for k in range(NBASE)]
    err_dp = _ddp_err(gt.ddPdrho.cpu().numpy(), ddp, gt.dPdrho.cpu().numpy(), _rate(st))
    print(name, "dbase row errors", ["%.1e" % e for e in errs], "ddPdrho %.1e" % err_dp)
    assert max(errs) < TAN_RTOL and err_dp < TAN_RTOL, (name, errs, err_dp)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the gradient
# ---------------------------------------------------------------------------------------------------------------------
def _points_fixture(D):
    gp = D["grad_points"]
    st = tables_from_fixture(D).select(gp[:, 0].astype(int))
    return st, gp[:, 1].copy(), gp[:, 2].copy(), D["theta"]


def _points_config5(npts=4096, nl=1025):
    from ideal_ballooning_solver_b200 import synthetic, tables
    rng = np.random.default_rng(20261018 + 5)
    s = rng.uniform(0.5, 0.95, npts); al = rng.uniform(0, np.pi, npts); t0 = rng.uniform(0, 0.5 * np.pi, npts)
    st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=1)).evaluate(s)
    return st, al, t0, np.linspace(-4 * np.pi, 4 * np.pi, nl)


def _grad_fd(dt, al, t0, theta, d, want_X=False):
    import torch
    from ideal_ballooning_solver_b200 import engine
    alphas = torch.from_numpy(np.stack([al - 0.5 * d, al, al + 0.5 * d], axis=1)).cuda()
    geo = engine.geometry_batch(dt, alphas, theta)
    return engine.obj_w_grad_batch(geo.base, geo.dPdrho, torch.from_numpy(t0).cuda(), engine.grid_spacing(theta), del_alpha=d,
                                   want_X=want_X)


def _grad_exact(dt, al, t0, theta, want_X=False):
    import torch
    from ideal_ballooning_solver_b200 import engine
    geo = engine.geometry_tangent_batch(dt, torch.from_numpy(al[:, None].copy()).cuda(), theta)
    return engine.obj_w_grad_tangent_batch(geo.base, geo.dbase, geo.dPdrho, geo.ddPdrho, torch.from_numpy(t0).cuda(),
                                           engine.grid_spacing(theta), want_X=want_X)


def _lam(dt, al, t0, theta):
    import torch
    from ideal_ballooning_solver_b200 import engine
    geo = engine.geometry_batch(dt, torch.from_numpy(al[:, None].copy()).cuda(), theta)
    sol = engine.solve_base_batch(geo.base, geo.dPdrho, torch.from_numpy(t0).cuda(), engine.grid_spacing(theta), nth0=1,
                                  want_X=False, want_dX=False, want_matrix=False)
    return sol.lam.cpu().numpy()


def _check_gradient(st, al, t0, theta, what, resolve=True):
    dt = _tables(st)
    v_fd, g_fd, X_fd, _, i_fd = _grad_fd(dt, al, t0, theta, 0.004, want_X=True)
    v, g, X, _, info = _grad_exact(dt, al, t0, theta, want_X=True)
    assert int(((info.cpu().numpy() >> 16) & 3).max()) == 0, what
    # the solve and the theta0 part are the three-line path's bits
    assert np.array_equal(v.cpu().numpy(), v_fd.cpu().numpy()), what
    assert np.array_equal(g[:, 1].cpu().numpy(), g_fd[:, 1].cpu().numpy()), what
    assert np.array_equal(X.cpu().numpy(), X_fd.cpu().numpy()), what
    assert np.array_equal(info.cpu().numpy(), i_fd.cpu().numpy()), what
    ga = g[:, 0].cpu().numpy()
    fd = {d: (g_fd if d == 0.004 else _grad_fd(dt, al, t0, theta, d)[1])[:, 0].cpu().numpy() for d in (0.004, 0.002, 0.001)}
    e = {d: np.abs(fd[d] - ga) for d in fd}
    scale = max(float(np.max(np.abs(ga))), 1e-300)
    big = e[0.004] > 1e-6 * scale                                    # points whose truncation error is far above rounding
    r1, r2 = ((np.median(e[0.004][big] / e[0.002][big]), np.median(e[0.002][big] / e[0.001][big])) if big.any()
              else (float("nan"), float("nan")))
    rich = (4 * fd[0.001] - fd[0.002]) / 3
    err_rich = float(np.max(np.abs(rich - ga)) / scale)
    print(what, "|FD(0.004) - exact| / max|exact|: max %.2e median %.2e; halving ratios %.2f %.2f; Richardson %.1e"
          % (np.max(e[0.004]) / scale, np.median(e[0.004]) / scale, r1, r2, err_rich))
    if big.any():
        assert 3.5 < r1 < 4.5 and 3.5 < r2 < 4.5, (what, r1, r2)
    else:
        # axisymmetric tables: alpha enters only through the secular term (phi - phi_c) iota' of grad alpha, so g and c are
        # polynomials of degree <= 2 in alpha and the central difference has no truncation error: it must agree to rounding
        assert not (np.any(st.xn) or np.any(st.xn_nyq)), what
        assert np.max(e[0.004]) <= 1e-9 * scale, what
    assert err_rich < 2e-9, (what, err_rich)
    if resolve:
        # against re-solved eigenvalues: Richardson central differences of lambda(alpha +- h); grad[:, 0] = -d lam / d alpha
        hh = 1e-3
        d1 = (_lam(dt, al + hh, t0, theta) - _lam(dt, al - hh, t0, theta)) / (2 * hh)
        d2 = (_lam(dt, al + hh / 2, t0, theta) - _lam(dt, al - hh / 2, t0, theta)) / hh
        dl = (4 * d2 - d1) / 3
        # The reference's Hellmann-Feynman contraction (utils.py:1676-1680, Simpson quadrature) is not exactly the derivative
        # of its own discrete eigenvalue; the three-line finite difference carries the same offset.  Measured on a B200: up to
        # 5.9e-3 of max |grad| (ncsx_wout_op), 2.4e-4 on the config-5 sample.
        err = float(np.max(np.abs(-dl - ga)) / scale)
        err_fd = float(np.max(np.abs(-dl - fd[0.004])) / scale)
        print(what, "against re-solved lambda: exact %.1e, fd %.1e" % (err, err_fd))
        assert err < 1e-2 and abs(err - err_fd) <= 2 * float(np.max(e[0.004])) / scale + 1e-12, (what, err, err_fd)


@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXTURES)
def test_gradient_on_fixtures(cuda_lib, golden, name):
    _check_gradient(*_points_fixture(golden(name)), name)


@pytest.mark.gpu
def test_gradient_config5_sample(cuda_lib):
    """4096 NCSX-like points with (s, alpha, theta0) i.i.d. uniform, N = 1025 (the adjoint configuration's seeds)."""
    _check_gradient(*_points_config5(), "config5")


@pytest.mark.gpu
def test_gradient_long_line_cluster_solver(cuda_lib):
    """N = 16 385: the solve is the cluster form of the team solver."""
    st, al, t0, _ = _points_config5(npts=16)
    _check_gradient(st, al, t0, np.linspace(-32 * np.pi, 32 * np.pi, 16385), "N=16385", resolve=False)


@pytest.mark.gpu
def test_deterministic(cuda_lib):
    st, al, t0, theta = _points_config5(npts=256)
    dt = _tables(st)
    a = [t.cpu().numpy() for t in _grad_exact(dt, al, t0, theta, want_X=True)]
    b = [t.cpu().numpy() for t in _grad_exact(dt, al, t0, theta, want_X=True)]
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    import torch
    from ideal_ballooning_solver_b200 import engine
    g1 = engine.geometry_tangent_batch(dt, torch.from_numpy(al[:, None].copy()).cuda(), theta)
    g2 = engine.geometry_tangent_batch(dt, torch.from_numpy(al[:, None].copy()).cuda(), theta)
    assert np.array_equal(g1.dbase.cpu().numpy(), g2.dbase.cpu().numpy())
    assert np.array_equal(g1.ddPdrho.cpu().numpy(), g2.ddPdrho.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------------
# GPU: refinement
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refine_with_exact_alpha_derivative(cuda_lib):
    """The 64-surface NCSX case of test_refine_batches_all_surfaces with alpha_derivative="exact": every surface succeeds, the
    maximum never drops below the coarse one, and it agrees with the finite-difference refinement."""
    from ideal_ballooning_solver_b200 import scan, synthetic, tables
    st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=4)).evaluate(np.linspace(0.5, 0.95, 64))
    theta = np.linspace(-4 * np.pi, 4 * np.pi, 513)
    res = scan.ball_scan(st, theta=theta, nalpha_guess=6, ntheta0_guess=5, alpha_derivative="exact")
    res_fd = scan.ball_scan(st, theta=theta, nalpha_guess=6, ntheta0_guess=5)
    assert np.all(res.refine.success)
    assert np.all(res.gamma >= res.gamma_coarse.reshape(64, -1).max(axis=1) - 1e-12)
    assert np.all(res.gamma >= res_fd.gamma - 1e-10 - 1e-6 * np.abs(res_fd.gamma))
    rel = np.abs(res.gamma - res_fd.gamma) / np.abs(res_fd.gamma)
    print("refine exact vs fd: median rel %.1e, max rel %.1e, rounds %d vs %d" % (np.median(rel), rel.max(), res.refine.nbatches,
                                                                               res_fd.refine.nbatches))
    assert np.median(rel) < 1e-6
