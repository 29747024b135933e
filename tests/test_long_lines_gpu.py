"""GPU: field lines longer than one CTA can hold (N > 8194) -- the team solver spread over a thread-block cluster.

1. The cluster form equals the single-CTA form on the same input (IBS_TEAM_CLUSTER forces it at small N).
2. Long s-alpha lines against the oracle's LAPACK route.
3. Long 3-D lines by size-independent properties (Sturm certificates, pencil residual, Simpson quotient, dX stencil).
4. The lane kernels against the team kernel above N = 8194.
5. The scan driver end to end on long lines; the gradient, host-scan and reference-API entry points.
6. The limit N = 65 538."""
import dataclasses
import os

import numpy as np
import pytest

from helpers import LAM_RTOL, X_ATOL, s_alpha_base, sign_normalise

pytestmark = pytest.mark.gpu

N_MAX = 65538
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def _engine():
    from ideal_ballooning_solver_b200 import engine
    return engine


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _simpson(N):
    """scipy.integrate.simpson weights, unit spacing (odd N: composite 1/3 rule)."""
    assert N % 2 == 1
    w = np.where(np.arange(N) % 2 == 1, 4.0 / 3.0, 2.0 / 3.0)
    w[0] = w[-1] = 1.0 / 3.0
    return w


def _forced(monkeypatch, C, fn):
    """fn() with every team-kernel batch on a cluster of C CTAs, then the knob cleared again."""
    monkeypatch.setenv("IBS_TEAM_CLUSTER", str(C))
    try:
        return fn()
    finally:
        monkeypatch.delenv("IBS_TEAM_CLUSTER")


# ---------------------------------------------------------------------------------------------------------------------
# 1. cluster form == single-CTA form
# ---------------------------------------------------------------------------------------------------------------------
def _same_solution(a, b, worst):
    import torch
    assert torch.equal(a.flags, b.flags)
    la, lb = a.lam.cpu().numpy(), b.lam.cpu().numpy()
    np.testing.assert_allclose(la, lb, rtol=LAM_RTOL, atol=0)
    worst["lam"] = max(worst["lam"], float(np.max(np.abs(la - lb) / np.abs(lb).clip(1e-300))))
    for name in ("X", "dX", "lam_matrix"):
        x, y = getattr(a, name), getattr(b, name)
        if x is None:
            continue
        d = float((x - y).abs().max().item())
        tol = X_ATOL * (float(y.abs().max().item()) if name == "dX" else 1.0)
        assert d <= tol, (name, d)
        worst[name] = max(worst.get(name, 0.0), d)


def _small_cases():
    """(label, callable) of team-kernel batches below N = 8194: every coefficient source, chained runs, count-only."""
    import torch
    from ideal_ballooning_solver_b200 import synthetic
    from helpers import fixture_gcf
    eng = _engine()
    cases = []
    G = _golden("s_alpha")
    for nth in (1024, 2048, 512):
        theta = G[f"theta_{nth}"]
        cs = G["cases"]
        g, c, f = (_cuda(a) for a in synthetic.s_alpha_coefficients(cs[:, 0], cs[:, 1], cs[:, 2], theta))
        sig = torch.full((len(cs),), 2.0, dtype=torch.float64)
        cases.append((f"s_alpha_{nth}", lambda g=g, c=c, f=f, h=eng.grid_spacing(theta), sig=sig:
                      eng.solve_gcf_batch(g, c, f, h, sigma=sig)))
    for name in ("synthetic_ncsx", "synthetic_d3d"):
        D = _golden(name)
        ns, na, nt = D["lam_conv"].shape
        gcf = [fixture_gcf(D, i, j, k) for i in range(ns) for j in range(na) for k in range(nt)]
        g, c, f = (_cuda(np.array([x[m] for x in gcf])) for m in range(3))
        cases.append((name, lambda g=g, c=c, f=f, h=eng.grid_spacing(D["theta"]): eng.solve_gcf_batch(g, c, f, h)))
    # base arrays of s-alpha lines: line_of_solve (exact coefficients), the polynomial path (nth0 >= 4, even N) and chains
    for N in (65, 700, 1025, 2048):
        theta = np.linspace(-6 * np.pi, 6 * np.pi, N)
        lines = [(0.8, 0.8), (1.2, 0.3), (0.4, 0.6)]
        bases = [s_alpha_base(sh, al, theta) for sh, al in lines]
        base = _cuda(np.stack([b for b, _ in bases]))
        dP = _cuda(np.array([d for _, d in bases]))
        nt = 16
        th0 = _cuda(np.tile(np.linspace(0.0, 0.5 * np.pi, nt), len(lines)))
        h = eng.grid_spacing(theta)
        line = torch.arange(len(lines), dtype=torch.int32).repeat_interleave(nt).cuda()
        cases.append((f"base_line_of_solve_{N}", lambda base=base, dP=dP, th0=th0, h=h, line=line:
                      eng.solve_base_batch(base, dP, th0, h, line_of_solve=line)))
        cases.append((f"base_line_of_solve_chain16_{N}", lambda base=base, dP=dP, th0=th0, h=h, line=line:
                      eng.solve_base_batch(base, dP, th0, h, line_of_solve=line, chain_len=16)))
        if N % 2 == 0:      # odd N with nth0 >= 4 goes to the lane kernels
            cases.append((f"base_poly_chain16_{N}", lambda base=base, dP=dP, th0=th0, h=h, nt=nt:
                          eng.solve_base_batch(base, dP, th0, h, nth0=nt, chain_len=16)))
            cases.append((f"base_poly_{N}", lambda base=base, dP=dP, th0=th0, h=h, nt=nt:
                          eng.solve_base_batch(base, dP, th0, h, nth0=nt)))
    return cases


@pytest.fixture(scope="module")
def small_cases(cuda_lib):
    return _small_cases()


@pytest.mark.parametrize("C", [2, 4, 8])
def test_cluster_form_equals_single_cta_form(cuda_lib, small_cases, monkeypatch, C):
    worst = {"lam": 0.0}
    for label, run in small_cases:
        ref = run()
        got = _forced(monkeypatch, C, run)
        try:
            _same_solution(got, ref, worst)
        except AssertionError as e:
            raise AssertionError(f"{label}: {e}") from e
    print(f"C = {C}: largest deviation cluster vs single CTA: {worst}")


@pytest.mark.parametrize("C", [2, 4, 8])
def test_cluster_count_above_equals_single_cta(cuda_lib, monkeypatch, C):
    import torch
    from scipy.linalg import eigh_tridiagonal
    from oracle import ballooning_oracle as bo
    from ideal_ballooning_solver_b200 import synthetic
    eng = _engine()
    rng = np.random.default_rng(3)
    for N in (65, 700, 1025):
        theta = np.linspace(-6 * np.pi, 6 * np.pi, N)
        g, c, f = synthetic.s_alpha_coefficients(0.7, 0.9, 0.1, theta)
        _, _, _, fu, sub, diag, sup = bo.discretise(theta, g, c, f)
        fi = fu[1:-1]
        ev = eigh_tridiagonal(diag, sup * np.sqrt(fi[:-1] / fi[1:]), eigvals_only=True)
        lam = np.concatenate([rng.uniform(ev[-20], ev[-1] + 0.1, 64), ev[-4:] + 1e-9, ev[-4:] - 1e-9])
        rep = lambda a: _cuda(np.tile(a, (len(lam), 1)))
        args = (rep(g), rep(c), rep(f), eng.grid_spacing(theta), _cuda(lam))
        ref = eng.count_above_batch(*args)
        got = _forced(monkeypatch, C, lambda: eng.count_above_batch(*args))
        assert torch.equal(got, ref)
        assert np.array_equal(got.cpu().numpy(), (ev[None, :] > lam[:, None]).sum(axis=1))


# ---------------------------------------------------------------------------------------------------------------------
# 2. long s-alpha lines against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [16385, 32769, 65537, 20000])
def test_long_s_alpha_lines_match_oracle(cuda_lib, N):
    """At these sizes the oracle's own accuracy is the limit: LAPACK's eigenvalue carries ~eps ||S|| (||S|| ~ max |diag|
    of the symmetrised pencil; test_solver_gpu.py allows 8 eps ||S||) and its eigenvector eps ||S|| / gap.  lambda must agree to LAM_RTOL or to that bound, X to
    X_ATOL wherever the oracle's eigenvector is itself good to 1e-9."""
    from oracle import ballooning_oracle as bo
    from ideal_ballooning_solver_b200 import synthetic
    eng = _engine()
    cases = _golden("s_alpha")["cases"]
    theta = np.linspace(-61 * np.pi, 61 * np.pi, N)
    g, c, f = synthetic.s_alpha_coefficients(cases[:, 0], cases[:, 1], cases[:, 2], theta)
    sol = eng.solve_gcf_batch(_cuda(g), _cuda(c), _cuda(f), eng.grid_spacing(theta))
    assert np.all(sol.flags.cpu().numpy() == 0), sol.info
    lam, X = sol.lam.cpu().numpy(), sol.X.cpu().numpy()
    assert np.all(X >= 0) and np.all(X.max(axis=1) == 1.0)
    one = np.ones(N)
    nx = 0
    for k in range(len(cases)):
        # dPdrho = -1, B = gradpar = 1: the reference forms g = gds2, c = cvdrift, f = gds2 (utils.py:1560-1562)
        info = {}
        lr, Xr, *_ = bo.gamma_ball_full(-1.0, theta, one, one, c[k], g[k], method="lambda_max", info=info)
        diag = bo.discretise(theta, g[k], c[k], f[k])[5]
        eps_s = 2.2e-16 * np.abs(diag).max()
        dx = float(np.max(np.abs(X[k] - sign_normalise(Xr))))
        x_cond = eps_s / info["gap"] if info["gap"] > 0 else np.inf
        print(f"N = {N} case {k}: lambda {lam[k]:+.6e} rel {abs(lam[k] - lr) / abs(lr):.1e} abs {abs(lam[k] - lr):.1e} "
              f"(eps||S|| {eps_s:.1e}), X {dx:.1e} (eps||S||/gap {x_cond:.1e})")
        assert (lam[k] > 0) == (lr > 0)
        assert abs(lam[k] - lr) <= max(LAM_RTOL * abs(lr), 8 * eps_s), k
        if x_cond <= 1e-9:
            assert dx < X_ATOL, (k, dx)
            nx += 1
    assert nx >= 3


# ---------------------------------------------------------------------------------------------------------------------
# 3. long 3-D lines by properties
# ---------------------------------------------------------------------------------------------------------------------
def _geo(kind, ns, na, nt, N, span, seed=11):
    import torch
    from ideal_ballooning_solver_b200 import synthetic, tables
    eng = _engine()
    st = tables.RadialSplines(synthetic.make_equilibrium(kind, seed=seed)).evaluate(np.linspace(0.5, 0.95, ns))
    theta = np.linspace(-span * np.pi, span * np.pi, N)
    geo = eng.geometry_batch(eng.DeviceTables.from_host(st), np.linspace(0.0, np.pi, na), theta, want_info=True)
    assert int((geo.info >> 16).max().item()) == 0
    th0 = torch.from_numpy(np.linspace(0.0, 0.5 * np.pi, nt)).cuda().repeat(ns * na)
    return st, geo, th0, theta


@pytest.mark.parametrize("kind", ["ncsx", "hberg"])
def test_long_3d_lines_properties(cuda_lib, kind):
    import torch
    eng = _engine()
    ns, na, nt, N = 3, 4, 4, 16385
    st, geo, th0, theta = _geo(kind, ns, na, nt, N, 16)
    h = eng.grid_spacing(theta)
    n = th0.numel()
    line = (torch.arange(n, device="cuda") // nt).to(torch.int32)
    ex = eng.solve_base_batch(geo.base, geo.dPdrho, th0, h, line_of_solve=line, want_gcf=True)
    assert int((ex.flags & 3).max().item()) == 0
    # X >= 0, max exactly 1, Dirichlet ends
    X = ex.X
    assert bool((X >= 0).all()) and bool((X.max(dim=1).values == 1.0).all())
    assert bool((X[:, 0] == 0).all()) and bool((X[:, -1] == 0).all())
    # bit-identical reruns; chained == independent
    ex2 = eng.solve_base_batch(geo.base, geo.dPdrho, th0, h, line_of_solve=line, want_gcf=True)
    for a, b in ((ex.lam, ex2.lam), (ex.X, ex2.X), (ex.dX, ex2.dX), (ex.info, ex2.info)):
        assert torch.equal(a, b)
    ch = eng.solve_base_batch(geo.base, geo.dPdrho, th0, h, line_of_solve=line, chain_len=16)
    rel = lambda a, b: float(((a - b).abs() / b.abs().clamp_min(1e-300)).max().item())
    assert rel(ch.lam, ex.lam) < 1e-11
    assert float((ch.X - ex.X).abs().max().item()) < 1e-9
    # Sturm certificates through the cluster count-only kernel
    g, c, f = ex.g, ex.c, ex.f
    lam_m = ex.lam_matrix
    scale = lam_m.abs().clamp_min(1e-3)
    cnt_hi = eng.count_above_batch(g, c, f, h, lam_m + 1e-9 * scale)
    cnt_lo = eng.count_above_batch(g, c, f, h, lam_m - 1e-7 * scale)
    assert int(cnt_hi.max().item()) == 0 and int(cnt_lo.min().item()) >= 1
    # residual of the discrete pencil (K - lam F) x on the interior rows (utils.py:1584-1592)
    gh = 0.5 * (g[:, 1:] + g[:, :-1])
    Kx = (gh[:, 1:] * (X[:, 2:] - X[:, 1:-1]) - gh[:, :-1] * (X[:, 1:-1] - X[:, :-2])) / h ** 2 + c[:, 1:-1] * X[:, 1:-1]
    res = Kx - lam_m[:, None] * f[:, 1:-1] * X[:, 1:-1]
    norm = (gh.abs().max(dim=1).values / h ** 2)[:, None]
    assert float((res.abs() / norm).max().item()) < 1e-11
    # the returned gam is the Simpson Rayleigh quotient of (X, dX) (utils.py:1618-1621)
    w = _cuda(_simpson(N))
    y0 = (w * (-g * ex.dX ** 2 + c * X ** 2)).sum(dim=1)
    y1 = (w * f * X ** 2).sum(dim=1)
    assert rel(ex.lam, y0 / y1) < 1e-9
    # dX is the reference stencil of X
    dX_ref = torch.zeros_like(X)
    dX_ref[:, 2:-2] = 2 / (3 * h) * (X[:, 3:-1] - X[:, 1:-3]) - (X[:, 4:] - X[:, :-4]) / (12 * h)
    dX_ref[:, 1] = (X[:, 2] - X[:, 0]) / (2 * h); dX_ref[:, -2] = (X[:, -1] - X[:, -3]) / (2 * h)
    dX_ref[:, 0] = (-1.5 * X[:, 0] + 2 * X[:, 1] - 0.5 * X[:, 2]) / h
    dX_ref[:, -1] = (0.5 * X[:, -3] - 2 * X[:, -2]) / h
    assert float((ex.dX - dX_ref).abs().max().item()) < 1e-10 / h


# ---------------------------------------------------------------------------------------------------------------------
# 4. lane kernels against the team kernel above N = 8194
# ---------------------------------------------------------------------------------------------------------------------
def test_lane_kernels_match_cluster_team_kernel(cuda_lib, monkeypatch):
    import torch
    from ideal_ballooning_solver_b200 import scan, synthetic, tables
    eng = _engine()
    st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=4)).evaluate(np.linspace(0.5, 0.95, 4))
    dt = eng.DeviceTables.from_host(st)
    theta = np.linspace(-8 * np.pi, 8 * np.pi, 16385)
    alpha, theta0 = np.linspace(0, np.pi, 6), np.linspace(0, 0.5 * np.pi, 8)
    lane = scan.coarse_scan(dt, alpha, theta0, theta, want_X=True)
    monkeypatch.setenv("IBS_SCAN", "0")
    team = scan.coarse_scan(dt, alpha, theta0, theta, want_X=True)
    monkeypatch.delenv("IBS_SCAN")
    assert int((lane.info >> 16).max().item()) == 0 and int((team.info >> 16).max().item()) == 0
    np.testing.assert_allclose(lane.gamma.cpu().numpy(), team.gamma.cpu().numpy(), rtol=LAM_RTOL, atol=0)
    assert float((lane.X - team.X).abs().max().item()) < X_ATOL
    assert torch.equal(lane.idx, team.idx)


# ---------------------------------------------------------------------------------------------------------------------
# 5. end to end
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ncsx_long(cuda_lib):
    from ideal_ballooning_solver_b200 import synthetic, tables
    st = tables.RadialSplines(synthetic.make_equilibrium("ncsx", seed=4)).evaluate(np.linspace(0.55, 0.9, 4))
    return st, np.linspace(-8 * np.pi, 8 * np.pi, 16385)


def test_ball_scan_on_long_lines(cuda_lib, ncsx_long):
    import torch
    from ideal_ballooning_solver_b200 import engine, scan
    st, theta = ncsx_long
    na, nt = 6, 5
    res = scan.ball_scan(st, theta=theta, nalpha_guess=na, ntheta0_guess=nt)
    r = res.refine
    assert r is not None and np.all(r.success)
    cmax = res.gamma_coarse.reshape(st.ns, -1).max(axis=1)
    assert np.all(res.gamma >= cmax - 1e-10 * np.abs(cmax))
    assert np.all(np.isfinite(res.gamma)) and res.X.shape == (st.ns, len(theta))
    # the final gamma is the objective at the optimum (one independent solve per surface)
    dt = engine.DeviceTables.from_host(st)
    geo = engine.geometry_batch(dt, torch.from_numpy(res.alpha[:, None].copy()).cuda(), theta)
    fun = engine.solve_base_batch(geo.base, geo.dPdrho, torch.from_numpy(res.theta0.copy()).cuda(), engine.grid_spacing(theta),
                                  nth0=1, want_X=False, want_dX=False, want_matrix=False).lam.cpu().numpy()
    np.testing.assert_allclose(res.gamma, fun, rtol=1e-12, atol=0)
    # the reference's optimiser on the same evaluations
    res_s = scan.ball_scan(st, theta=theta, nalpha_guess=na, ntheta0_guess=nt, refine_method="scipy")
    np.testing.assert_allclose(res_s.gamma_coarse, res.gamma_coarse, rtol=0, atol=0)
    assert np.all(res.gamma >= res_s.gamma - 1e-10 - 1e-6 * np.abs(res_s.gamma))
    assert np.median(np.abs(res.gamma - res_s.gamma) / np.abs(res_s.gamma)) < 1e-6


def test_table_gradient_on_long_lines(cuda_lib, ncsx_long):
    import torch
    from ideal_ballooning_solver_b200 import engine, scan
    st, theta = ncsx_long
    rng = np.random.default_rng(5)
    a_star, t_star = rng.uniform(0.2, 2.5, st.ns), rng.uniform(0.0, 1.2, st.ns)
    dt0 = engine.DeviceTables.from_host(st)
    tg = scan.table_gradient(dt0, a_star, t_star, theta, scalars=True)
    h = engine.grid_spacing(theta)
    a = torch.from_numpy(a_star[:, None].copy()).cuda()
    t0 = torch.from_numpy(t_star.copy()).cuda()

    def lam_of(dt):
        geo = engine.geometry_batch(dt, a, theta)
        return engine.solve_base_batch(geo.base, geo.dPdrho, t0, h, nth0=1, want_X=False, want_dX=False,
                                       want_matrix=False).lam.cpu().numpy()

    np.testing.assert_allclose(tg.gamma, lam_of(dt0), rtol=1e-12)
    gmn, gnq, gsc = tg.grad_mn.cpu().numpy(), tg.grad_nyq.cpu().numpy(), tg.grad_scal.cpu().numpy()
    for (which, row, mode) in (("mn", 0, 0), ("mn", 0, 1), ("nyq", 1, 0), ("nyq", 0, 0)):
        base_tab = st.tab_mn if which == "mn" else st.tab_nyq
        step = max(1e-6 * np.abs(base_tab[:, row, mode]).max(), 5e-6)
        tp, tm = base_tab.copy(), base_tab.copy()
        tp[:, row, mode] += step; tm[:, row, mode] -= step
        key = "tab_mn" if which == "mn" else "tab_nyq"
        fd = (lam_of(engine.DeviceTables.from_host(dataclasses.replace(st, **{key: tp})))
              - lam_of(engine.DeviceTables.from_host(dataclasses.replace(st, **{key: tm})))) / (2 * step)
        ana = (gmn if which == "mn" else gnq)[:, row, mode]
        np.testing.assert_allclose(ana, fd, rtol=1e-2, atol=5e-3 * np.abs(fd).max() + 1e-12, err_msg=f"{which} {row} {mode}")
    # iota (scal column 1)
    step = 1e-5 * float(np.abs(st.scal[:, 1]).max())
    sp, sm = dt0.scal.clone(), dt0.scal.clone()
    sp[:, 1] += step; sm[:, 1] -= step
    fd = (lam_of(dataclasses.replace(dt0, scal=sp)) - lam_of(dataclasses.replace(dt0, scal=sm))) / (2 * step)
    np.testing.assert_allclose(gsc[:, 1], fd, rtol=1e-2, atol=5e-3 * np.abs(fd).max() + 1e-12, err_msg="iota")


def test_scan_host_xbest_on_long_lines(cuda_lib, ncsx_long):
    from ideal_ballooning_solver_b200 import engine, scan
    st, theta = ncsx_long
    alpha, theta0 = np.linspace(0, np.pi, 4), np.linspace(0, 0.5 * np.pi, 4)
    gamma, val, idx, sig, nbad, xbest = engine.scan_host(st, alpha, theta0, theta, want_xbest=True)
    assert nbad == 0
    cs = scan.coarse_scan(engine.DeviceTables.from_host(st), alpha, theta0, theta, want_X=True)
    np.testing.assert_array_equal(gamma, cs.gamma.cpu().numpy())
    np.testing.assert_array_equal(idx, cs.idx.cpu().numpy())
    Xc = cs.X.cpu().numpy().reshape(st.ns, -1, len(theta))
    for js in range(st.ns):
        # re-solved at the maximum by the team kernel (a cluster at this N): the same eigenfunction to rounding
        np.testing.assert_allclose(xbest[js], Xc[js, idx[js]], rtol=0, atol=X_ATOL)


def test_reference_api_gamma_ball_full_long_line(cuda_lib):
    from oracle import ballooning_oracle as bo
    from ideal_ballooning_solver_b200 import reference_api, synthetic
    N = 16385
    theta = np.linspace(-61 * np.pi, 61 * np.pi, N)
    g, c, _ = synthetic.s_alpha_coefficients(0.8, 0.8, 0.0, theta)
    one = np.ones(N)
    gam, X, dX, *_ = reference_api.gamma_ball_full(-1.0, theta, one, one, c, g)
    lr, Xr, *_ = bo.gamma_ball_full(-1.0, theta, one, one, c, g, method="lambda_max")
    np.testing.assert_allclose(gam, lr, rtol=LAM_RTOL, atol=0)
    np.testing.assert_allclose(sign_normalise(X), sign_normalise(Xr), rtol=0, atol=X_ATOL)


# ---------------------------------------------------------------------------------------------------------------------
# 6. the limit
# ---------------------------------------------------------------------------------------------------------------------
def test_longer_than_limit_is_refused(cuda_lib):
    import torch
    eng = _engine()
    N = N_MAX + 1
    g = torch.ones((1, N), dtype=torch.float64, device="cuda")
    with pytest.raises(RuntimeError, match="65538"):
        eng.solve_gcf_batch(g, g, g, 0.01)
    with pytest.raises(RuntimeError, match="65538"):
        eng.count_above_batch(g, g, g, 0.01, torch.zeros(1, dtype=torch.float64))
    # the longest accepted line still solves
    from ideal_ballooning_solver_b200 import synthetic
    theta = np.linspace(-61 * np.pi, 61 * np.pi, N_MAX)
    g, c, f = synthetic.s_alpha_coefficients(0.8, 0.8, 0.0, theta)
    sol = eng.solve_gcf_batch(_cuda(g[None]), _cuda(c[None]), _cuda(f[None]), eng.grid_spacing(theta))
    assert int(sol.flags.max().item()) == 0
