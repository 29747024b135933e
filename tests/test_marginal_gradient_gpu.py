"""First-order response of the critical pressure-gradient factor kappa*: the alpha-tangent entry point
(``ibs_marginal_tangent_batch``), the per-point sensitivities (``ibs_marginal_sensitivities``), ``scan.marginal_gradient`` (the
reverse mode of K1 on the kappa*-scaled tables) and ``scan.refine_marginal``.

Argument checks without a GPU; on the GPU: bit identity with ``marginal_batch``, d kappa*/d alpha against Richardson central
differences through K1, the table and scalar gradients against central differences of kappa* on perturbed tables, the scale
identity of p', the refinement against the coarse grid and against scipy's L-BFGS-B, and first-order prediction of the refined
minimum for perturbed equilibria."""
import copy
import dataclasses

import numpy as np
import pytest

from helpers import tables_from_fixture

FIXTURES = ["ncsx_wout_op", "synthetic_ncsx", "synthetic_d3d", "synthetic_hberg"]
THETA0 = np.array([0.0, 0.3, 0.9])
THETA = np.linspace(-3 * np.pi, 3 * np.pi, 513)


def _args_tangent(p, N=65, h=0.1, nsolve=4, nth0=1, kmax=1e3, rtol=1e-12, base=None, dbase=None, ddp=None, kappa=None, grad=None):
    d = lambda x: p if x is None else (None if x == 0 else x)
    return (d(base), d(dbase), p, d(ddp), p, None, nth0, nsolve, N, h, kmax, rtol, d(kappa), d(grad), None, None, None)


def test_argument_errors_without_gpu():
    """Both entry points reject bad sizes and null pointers before any CUDA call, with a message; empty batches return 0."""
    from ideal_ballooning_solver_b200 import _lib, build
    build.build()
    lib = _lib.load()
    buf = np.zeros(64)
    p = buf.ctypes.data

    def tan(**kw):
        return lib.ibs_marginal_tangent_batch(*_args_tangent(p, **kw))
    assert tan(nsolve=0) == 0
    assert tan(nsolve=-1) == 1 and b"5 <= N" in lib.ibs_last_error()
    assert tan(N=4) == 1 and b"5 <= N" in lib.ibs_last_error()
    assert tan(N=65539) == 1 and b"5 <= N" in lib.ibs_last_error()
    for kw in ("base", "dbase", "ddp", "kappa", "grad"):
        assert tan(**{kw: 0}) == 1 and b"null" in lib.ibs_last_error(), kw
    assert tan(nth0=0) == 1 and b"nth0" in lib.ibs_last_error()
    assert tan(h=0.0) == 1 and b"h must" in lib.ibs_last_error()
    assert tan(kmax=0.0) == 1 and b"kappa_max" in lib.ibs_last_error()
    assert tan(rtol=1.0) == 1 and b"rtol" in lib.ibs_last_error()

    def sens(nsolve=4, N=65, h=0.1, nth0=1, base=p, kappa=p, X=p, dg=p, dc=p):
        return lib.ibs_marginal_sensitivities(base, p, p, None, nth0, nsolve, N, h, kappa, X, dg, dc, None)
    assert sens(nsolve=0) == 0
    assert sens(nsolve=-1) == 1 and b"5 <= N" in lib.ibs_last_error()
    assert sens(N=4) == 1 and b"5 <= N" in lib.ibs_last_error()
    for kw in ("base", "kappa", "X", "dg", "dc"):
        assert sens(**{kw: None}) == 1 and b"null" in lib.ibs_last_error(), kw
    assert sens(nth0=0) == 1 and b"nth0" in lib.ibs_last_error()
    assert sens(h=-1.0) == 1 and b"h must" in lib.ibs_last_error()


# ---------------------------------------------------------------------------------------------------------------------
def _fixture_lines(D):
    """K1 and its alpha-tangent on the fixture's tables and alphas: (geometry, h) with lines flattened (ns * nalpha)."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    dt = engine.DeviceTables.from_host(tables_from_fixture(D))
    geo = engine.geometry_tangent_batch(dt, torch.from_numpy(np.asarray(D["alphas"], dtype=np.float64)).cuda(), D["theta"])
    return dt, geo, engine.grid_spacing(D["theta"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXTURES)
def test_tangent_bits_identical_to_marginal_batch(cuda_lib, golden, name):
    import torch
    from ideal_ballooning_solver_b200 import engine
    D = golden(name)
    _, geo, h = _fixture_lines(D)
    N = geo.base.shape[-1]
    base, dbase = geo.base.reshape(-1, 8, N), geo.dbase.reshape(-1, 8, N)
    dP, ddP = geo.dPdrho.reshape(-1), geo.ddPdrho.reshape(-1)
    nl, nt = base.shape[0], len(THETA0)
    th0 = torch.from_numpy(np.tile(THETA0, nl)).cuda()
    los = torch.from_numpy(np.random.default_rng(3).integers(0, nl, 2 * nl * nt)).cuda()
    th0_los = torch.from_numpy(np.random.default_rng(4).uniform(0, 1.5, los.numel())).cuda()
    for kw, t0 in ((dict(nth0=nt), th0), (dict(line_of_solve=los), th0_los)):
        m = engine.marginal_batch(base, dP, t0, h, want_X=True, want_derivs=True, **kw)
        mt = engine.marginal_tangent_batch(base, dbase, dP, ddP, t0, h, want_X=True, **kw)
        assert int((m.flags & 3).max().item()) == 0
        for f in ("kappa", "X", "info"):
            assert torch.equal(getattr(m, f), getattr(mt, f)), (name, f)
        assert torch.equal(m.dkappa_dtheta0, mt.grad[:, 1].contiguous()), name
        assert bool(torch.isfinite(mt.grad).all())
        # without X_out the same bits
        mt2 = engine.marginal_tangent_batch(base, dbase, dP, ddP, t0, h, **kw)
        assert torch.equal(mt2.kappa, mt.kappa) and torch.equal(mt2.grad, mt.grad) and torch.equal(mt2.info, mt.info)


def _kappa_k1(dt, alpha, t0, theta, **kw):
    """kappa* through the whole forward path: K1 on (alpha (ns,), theta0 (ns,)) one line per surface, then marginal_batch."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    a = torch.as_tensor(np.asarray(alpha, dtype=np.float64).reshape(-1, 1)).cuda()
    geo = engine.geometry_batch(dt, a, theta)
    return engine.marginal_batch(geo.base, geo.dPdrho, torch.as_tensor(np.asarray(t0, dtype=np.float64)).cuda(),
                                 engine.grid_spacing(theta), nth0=1, **kw).kappa.cpu().numpy()


def _richardson(fun, d):
    d1 = (fun(d) - fun(-d)) / (2 * d)
    d2 = (fun(d / 2) - fun(-d / 2)) / d
    return (4 * d2 - d1) / 3


@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXTURES)
def test_dkappa_dalpha_against_k1(cuda_lib, golden, name):
    """d kappa*/d alpha against Richardson central differences of kappa* through K1 (alpha -+ delta, delta and delta / 2), to 1e-7
    of the batch's largest |d kappa*/d alpha|.  On axisymmetric tables a shift of alpha is a shift of the secular term of grad
    alpha, i.e. a shift of theta0: there d kappa*/d alpha = -+ d kappa*/d theta0, with one sign for the whole batch."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    D = golden(name)
    dt = engine.DeviceTables.from_host(tables_from_fixture(D))
    theta = D["theta"]
    ns = dt.ns
    rng = np.random.default_rng(21)
    al = np.repeat(rng.uniform(0.1, 3.0, ns), len(THETA0))
    t0 = np.tile(THETA0, ns)
    dts = engine.DeviceTables(dt.tab_mn.repeat_interleave(len(THETA0), 0), dt.tab_nyq.repeat_interleave(len(THETA0), 0),
                              dt.scal.repeat_interleave(len(THETA0), 0), dt.xm, dt.xn, dt.xm_nyq, dt.xn_nyq, dt.phiedge, dt.Aminor_p)
    geo = engine.geometry_tangent_batch(dts, torch.from_numpy(al[:, None].copy()).cuda(), theta)
    mt = engine.marginal_tangent_batch(geo.base, geo.dbase, geo.dPdrho, geo.ddPdrho, torch.from_numpy(t0).cuda(),
                                       engine.grid_spacing(theta), nth0=1)
    assert int((mt.flags & 3).max().item()) == 0 and bool(torch.isfinite(mt.kappa).all())
    ga = mt.grad[:, 0].cpu().numpy()
    fd = _richardson(lambda d: _kappa_k1(dts, al + d, t0, theta), 1e-3)
    scale = np.abs(ga).max()
    err = np.abs(ga - fd).max() / scale
    print(f"{name}: max |d kappa*/d alpha| {scale:.3e}, error against K1 differences {err:.1e}")
    assert err <= 1e-7, (name, err)
    if not (np.any(dt.xn) or np.any(dt.xn_nyq)):
        gt = mt.grad[:, 1].cpu().numpy()
        e_plus, e_minus = np.abs(ga - gt).max(), np.abs(ga + gt).max()
        print(f"{name}: axisymmetric, |da - dt| {e_plus:.1e}, |da + dt| {e_minus:.1e}")
        assert min(e_plus, e_minus) <= 1e-8 * max(scale, np.abs(gt).max()), (e_plus, e_minus)


# ---------------------------------------------------------------------------------------------------------------------
def _lines(st, seed=5):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.2, 2.5, st.ns), rng.uniform(0.0, 1.2, st.ns)


def _with(dt, which, k, delta):
    """Copy of device tables with entry k of ``which`` (tab_mn row/mode, tab_nyq row/mode, scal column, or a global) moved by
    delta (per surface for the tables and scal)."""
    import torch
    if which in ("tab_mn", "tab_nyq"):
        t = getattr(dt, which).clone()
        t[:, k[0], k[1]] += torch.as_tensor(delta).cuda()
        return dataclasses.replace(dt, **{which: t})
    if which == "scal":
        t = dt.scal.clone()
        t[:, k] += torch.as_tensor(delta).cuda()
        return dataclasses.replace(dt, scal=t)
    return dataclasses.replace(dt, **{which: getattr(dt, which) + float(delta)})


@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXTURES)
def test_table_gradient_against_central_differences(cuda_lib, golden, name):
    """d kappa*/d (single Fourier coefficients of both tables, every scalar column, phiedge, Aminor_p) at fixed (alpha, theta0)
    against Richardson central differences of kappa* (K1 + marginal_batch on the perturbed tables), to 1e-6 of the surface's
    largest gradient entry; and p' d kappa*/d p' = -kappa*."""
    from ideal_ballooning_solver_b200 import engine, scan
    st = tables_from_fixture(golden(name))
    a_star, t_star = _lines(st)
    dt = engine.DeviceTables.from_host(st)
    mg = scan.marginal_gradient(dt, a_star, t_star, THETA, scalars=True)
    assert np.all(mg.finite)
    np.testing.assert_array_equal(mg.kappa, _kappa_k1(dt, a_star, t_star, THETA))
    gmn, gnq, gsc, ggl = (g.cpu().numpy() for g in (mg.grad_mn, mg.grad_nyq, mg.grad_scal, mg.grad_glob))
    for g in (gmn, gnq, gsc, ggl):
        assert np.all(np.isfinite(g))
    big = np.maximum(np.maximum(np.abs(gmn).reshape(st.ns, -1).max(1), np.abs(gnq).reshape(st.ns, -1).max(1)),
                     np.maximum(np.abs(gsc).max(1), np.abs(ggl).max(1)))
    # p' scale identity: kappa*(t p') = kappa*(p') / t
    np.testing.assert_allclose(gsc[:, 3] * st.scal[:, 3], -mg.kappa, rtol=1e-9)
    assert np.all(gsc[:, 5:] == 0.0)
    cases = []
    mn, mq = st.tab_mn.shape[2], st.tab_nyq.shape[2]
    for r in range(6):
        for q in sorted({0, 1, mn // 2, mn - 1}):
            cases.append(("tab_mn", (r, q), gmn[:, r, q], st.tab_mn[:, r, :]))
    for r in range(7):
        for q in sorted({0, 1, mq // 2, mq - 1}):
            cases.append(("tab_nyq", (r, q), gnq[:, r, q], st.tab_nyq[:, r, :]))
    for c in range(5):
        cases.append(("scal", c, gsc[:, c], st.scal[:, c:c + 1]))
    cases.append(("phiedge", None, ggl[:, 0], np.full((st.ns, 1), st.phiedge)))
    cases.append(("Aminor_p", None, ggl[:, 1], np.full((st.ns, 1), st.Aminor_p)))
    worst = 0.0
    for which, k, an, ref in cases:
        step = 1e-4 * np.abs(ref).max(axis=1)
        step = np.where(step > 0, step, 1e-4)
        if which in ("phiedge", "Aminor_p"):
            step = float(step[0])
        fd = _richardson(lambda d: _kappa_k1(_with(dt, which, k, d * step), a_star, t_star, THETA), 1.0) / step
        err = np.abs(an - fd) / big
        worst = max(worst, float(err.max()))
        assert np.all(err <= 1e-6), (name, which, k, an, fd)
    print(f"{name}: {len(cases)} directions, worst error {worst:.1e} of the largest entry")


@pytest.mark.gpu
def test_zero_pressure_gradient_surface(cuda_lib, golden):
    """A surface with p' = 0 is never unstable: kappa* = inf, finite False, and its gradient rows are 0 (no NaN)."""
    from ideal_ballooning_solver_b200 import engine, scan
    st = tables_from_fixture(golden("synthetic_ncsx"))
    st.scal[1, 3] = 0.0
    a_star, t_star = _lines(st)
    mg = scan.marginal_gradient(engine.DeviceTables.from_host(st), a_star, t_star, THETA, scalars=True)
    assert mg.kappa[1] == np.inf and not mg.finite[1] and mg.finite[0] and mg.finite[2]
    for g in (mg.grad_mn, mg.grad_nyq, mg.grad_scal, mg.grad_glob):
        g = g.cpu().numpy()
        assert np.all(np.isfinite(g)) and np.all(g[1] == 0.0) and np.any(g[0] != 0.0)
    dk_dg, dk_dc = engine.marginal_sensitivities(*_one_line_solve(st, a_star, t_star))
    assert bool(dk_dg[1].isnan().all()) and bool(dk_dc[1].isnan().all()) and bool(dk_dg[0].isfinite().all())


def _one_line_solve(st, a_star, t_star):
    import torch
    from ideal_ballooning_solver_b200 import engine
    geo = engine.geometry_batch(engine.DeviceTables.from_host(st), torch.from_numpy(a_star[:, None].copy()).cuda(), THETA)
    t0 = torch.from_numpy(t_star.copy()).cuda()
    h = engine.grid_spacing(THETA)
    m = engine.marginal_batch(geo.base, geo.dPdrho, t0, h, nth0=1, want_X=True)
    return geo.base, geo.dPdrho, t0, h, m.kappa, m.X


# ---------------------------------------------------------------------------------------------------------------------
ALPHA_GRID, THETA0_GRID = np.linspace(0.0, np.pi, 6), np.linspace(0.0, 0.5 * np.pi, 5)


def _ncsx(seed=4, ns=12, pert=None, eps=0.0):
    from ideal_ballooning_solver_b200 import engine, synthetic, tables
    w = synthetic.make_equilibrium("ncsx", seed=seed)
    if pert is not None:
        w = pert(w, eps)
    return engine.DeviceTables.from_host(tables.RadialSplines(w).evaluate(np.linspace(0.5, 0.9, ns)))


def _scipy_min(dt, a0, t0, bounds, opts):
    """scipy L-BFGS-B on kappa*(alpha, theta0) of each surface, with the device's objective and gradient."""
    import torch
    from scipy.optimize import minimize
    from ideal_ballooning_solver_b200 import engine
    h = engine.grid_spacing(THETA)
    out = []
    for i in range(dt.ns):
        sub = dataclasses.replace(dt, tab_mn=dt.tab_mn[i:i + 1].contiguous(), tab_nyq=dt.tab_nyq[i:i + 1].contiguous(),
                                  scal=dt.scal[i:i + 1].contiguous())

        def fun(x):
            geo = engine.geometry_tangent_batch(sub, torch.tensor([[x[0]]], dtype=torch.float64).cuda(), THETA)
            m = engine.marginal_tangent_batch(geo.base, geo.dbase, geo.dPdrho, geo.ddPdrho,
                                              torch.tensor([x[1]], dtype=torch.float64).cuda(), h, nth0=1)
            k = float(m.kappa[0].item())
            g = m.grad[0].cpu().numpy()
            return (k, g) if np.isfinite(k) else (1e300, np.zeros(2))
        out.append(minimize(fun, x0=(a0[i], t0[i]), jac=True, method="L-BFGS-B", bounds=bounds, options=opts).fun)
    return np.array(out)


@pytest.mark.gpu
def test_refine_marginal(cuda_lib):
    """Every finite surface ends at or below its coarse minimum and at or below scipy's L-BFGS-B from the same start with the
    same objective, gradient, bounds and options; a surface with p' = 0 (kappa* = inf everywhere) passes through unchanged."""
    from ideal_ballooning_solver_b200 import scan
    dt = _ncsx()
    sc = dt.scal.clone()
    sc[3, 3] = 0.0
    dt = dataclasses.replace(dt, scal=sc)
    ms = scan.marginal_scan(dt, ALPHA_GRID, THETA0_GRID, THETA)
    r = scan.refine_marginal(dt, ms.alpha_crit, ms.theta0_crit, THETA)
    kc = ms.kappa_min.cpu().numpy()
    a0, t0 = ms.alpha_crit.cpu().numpy(), ms.theta0_crit.cpu().numpy()
    fin = np.isfinite(kc)
    assert not fin[3] and fin.sum() == dt.ns - 1
    assert r.fun[3] == kc[3] and r.alpha[3] == a0[3] and r.theta0[3] == t0[3] and not r.success[3]
    assert np.all(r.success[fin])
    assert np.all(r.fun[fin] <= kc[fin] * (1 + 2.3e-16))
    bounds = ((0.0, np.pi), (0.0, 0.5 * np.pi))
    ks = _scipy_min(dt, a0, t0, bounds, {"ftol": 5e-11, "gtol": 2e-8, "maxiter": 30})
    print("refine_marginal: coarse", kc[fin], "device", r.fun[fin], "scipy", ks[fin], "rounds", r.nbatches)
    assert np.all(r.fun[fin] <= ks[fin] + 1e-10 * ks[fin]), (r.fun[fin] - ks[fin])


def _pert_profiles(w, eps):
    wp = copy.copy(w)
    s_full = np.linspace(0.0, 1.0, w.ns)
    s_half = np.concatenate([[0.0], s_full[1:] - 0.5 * (s_full[1] - s_full[0])])
    wp.iotas = w.iotas * (1.0 + eps * (1.0 + s_half))
    wp.pres = w.pres * (1.0 + 0.5 * eps * (1.0 - s_half))
    return wp


def _pert_fourier(w, eps):
    wp = copy.copy(w)
    rng = np.random.default_rng(7)
    wp.rmnc = w.rmnc * (1.0 + eps * rng.standard_normal(w.rmnc.shape[0])[:, None] * np.exp(-0.3 * np.arange(w.rmnc.shape[0]))[:, None])
    return wp


def _kappa_min(dt):
    from ideal_ballooning_solver_b200 import scan
    ms = scan.marginal_scan(dt, ALPHA_GRID, THETA0_GRID, THETA)
    r = scan.refine_marginal(dt, ms.alpha_crit, ms.theta0_crit, THETA)
    assert np.all(r.success)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["profiles", "fourier"])
def test_first_order_end_to_end(cuda_lib, kind):
    """marginal_gradient(...).predict at the refined minimum against a re-run marginal_scan + refine_marginal on the perturbed
    equilibrium: the error falls at second order (ratio ~4 when eps halves)."""
    from ideal_ballooning_solver_b200 import scan
    pert = _pert_profiles if kind == "profiles" else _pert_fourier
    dt0 = _ncsx(seed=11, ns=6)
    r0 = _kappa_min(dt0)
    mg = scan.marginal_gradient(dt0, r0.alpha, r0.theta0, THETA, scalars=True)
    np.testing.assert_allclose(mg.kappa, r0.fun, rtol=1e-14)
    errs = []
    for eps in (2e-3, 1e-3):
        dtp = _ncsx(seed=11, ns=6, pert=pert, eps=eps)
        pred = mg.predict(dt0, [dtp])[0]
        actual = _kappa_min(dtp).fun - r0.fun
        errs.append(np.abs(pred - actual))
        print(kind, eps, "actual", actual, "error", errs[-1])
        assert np.median(np.abs(actual) / errs[-1]) > 10
    ratio = np.median(errs[0] / errs[1])
    print(kind, "halving ratio", errs[0] / errs[1])
    assert 3.0 < ratio < 5.0, ratio
