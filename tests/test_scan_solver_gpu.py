"""GPU parity of the lane kernels of the scan solver (ibs_scan_solver.cu: scan2_solve_kernel, and scan_solve_kernel with
IBS_SCAN2=0 or for grids scan2 cannot take) -- through the C ABI -- against the oracle, the stored converged-reference
values and the team-per-solve kernel (IBS_SCAN=0)."""
import os

import numpy as np
import pytest

from helpers import LAM_RTOL, X_ATOL, fixture_base, s_alpha_base, sign_normalise

pytestmark = pytest.mark.gpu


def _solve(base, dP, th0, h, nth0, scan, scan2=True, **kw):
    from ideal_ballooning_solver_b200 import engine
    old = {k: os.environ.get(k) for k in ("IBS_SCAN", "IBS_SCAN2")}
    os.environ["IBS_SCAN"] = "1" if scan else "0"
    os.environ["IBS_SCAN2"] = "1" if scan2 else "0"
    try:
        return engine.solve_base_batch(base, dP, th0, h, nth0=nth0, **kw)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.mark.parametrize("name", ["synthetic_d3d", "synthetic_ncsx", "synthetic_hberg", "ncsx_wout_op"])
@pytest.mark.parametrize("nth0", [5, 37, 70, 64])
@pytest.mark.parametrize("scan2", [True, False], ids=["scan2", "scan"])
def test_scan_kernel_matches_team_kernel_and_oracle(cuda_lib, golden, name, nth0, scan2):
    import torch
    from ideal_ballooning_solver_b200 import engine
    from oracle import ballooning_oracle as bo
    D = golden(name)
    theta = D["theta"]
    if (len(theta) & 1) == 0 or len(theta) < 65:
        pytest.skip("scan kernel needs an odd number of points")
    h = engine.grid_spacing(theta)
    fb = fixture_base(D)
    ns, na = fb.shape[:2]
    base = torch.from_numpy(fb).cuda()
    dP = torch.from_numpy(D["dPdrho"]).cuda()
    t0 = np.linspace(0.0, np.pi / 2, nth0)
    th0 = torch.from_numpy(np.tile(t0, ns * na)).cuda()
    sigma = torch.full((th0.numel(),), 1.0, dtype=torch.float64)
    new = _solve(base, dP, th0, h, nth0, True, scan2, sigma=sigma)
    old = _solve(base, dP, th0, h, nth0, False, sigma=sigma)
    assert np.all(new.flags.cpu().numpy() == old.flags.cpu().numpy())
    lam_n, lam_o = new.lam.cpu().numpy(), old.lam.cpu().numpy()
    np.testing.assert_allclose(lam_n, lam_o, rtol=LAM_RTOL, atol=0)
    assert np.array_equal(lam_n > 0, lam_o > 0)
    np.testing.assert_allclose(new.lam_matrix.cpu().numpy(), old.lam_matrix.cpu().numpy(), rtol=LAM_RTOL, atol=0)
    Xn, Xo = new.X.cpu().numpy(), old.X.cpu().numpy()
    np.testing.assert_allclose(Xn, Xo, rtol=0, atol=X_ATOL)
    assert np.all(Xn.max(axis=1) == 1.0) and np.all(Xn[:, 0] == 0) and np.all(Xn[:, -1] == 0)
    dXn, dXo = new.dX.cpu().numpy(), old.dX.cpu().numpy()
    np.testing.assert_allclose(dXn, dXo, rtol=0, atol=10 * X_ATOL * max(1.0, np.abs(dXo).max()))
    assert new.iterations.max().item() < 64
    # a sample against the oracle (LAPACK on the same pencil + the reference's post-processing)
    rng = np.random.default_rng(7)
    for s in rng.choice(th0.numel(), size=4, replace=False):
        line, t = divmod(int(s), nth0)
        i, j = divmod(line, na)
        cv = D["geo_cvdrift"][i, j] + t0[t] * D["geo_cvdrift0"][i, j]
        gd = D["geo_gds2"][i, j] + 2 * t0[t] * D["geo_gds21"][i, j] + t0[t] ** 2 * D["geo_gds22"][i, j]
        gam, X, dX, *_ = bo.gamma_ball_full(D["dPdrho"][i, j], theta, D["geo_bmag"][i, j], D["geo_gradpar_theta_pest"][i, j],
                                            cv, gd, method="lambda_max")
        assert abs(lam_n[s] - gam) <= LAM_RTOL * abs(gam)
        np.testing.assert_allclose(Xn[s], sign_normalise(X), rtol=0, atol=X_ATOL)


def test_scan_kernel_fixture_values(cuda_lib, golden):
    """Stored converged-reference eigenvalues (the reference itself, ARPACK tol=0) at the fixture's theta0, padded to a
    scan-shaped batch."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    D = golden("synthetic_ncsx")
    theta = D["theta"]
    h = engine.grid_spacing(theta)
    fb = fixture_base(D)
    ns, na = fb.shape[:2]
    t0 = np.concatenate([D["theta0s"], np.linspace(0.05, 1.5, 6)])
    nt = len(D["theta0s"])
    th0 = torch.from_numpy(np.tile(t0, ns * na)).cuda()
    sol = _solve(torch.from_numpy(fb).cuda(), torch.from_numpy(D["dPdrho"]).cuda(), th0, h, len(t0), True)
    lam = sol.lam.cpu().numpy().reshape(ns, na, len(t0))[:, :, :nt]
    np.testing.assert_allclose(lam, D["lam_conv"], rtol=LAM_RTOL, atol=0)
    X = sol.X.cpu().numpy().reshape(ns, na, len(t0), -1)[:, :, :nt]
    np.testing.assert_allclose(X, sign_normalise(D["X_conv"]), rtol=0, atol=X_ATOL)


def test_scan_kernel_outputs_optional_and_bad_input(cuda_lib, golden):
    import torch
    from ideal_ballooning_solver_b200 import engine
    D = golden("synthetic_d3d")
    theta = D["theta"]
    h = engine.grid_spacing(theta)
    fb = fixture_base(D).reshape(-1, 8, len(theta))[:2].copy()
    fb[1, 4, 100] = np.nan
    th0 = torch.from_numpy(np.tile(np.linspace(0, 1.2, 9), 2)).cuda()
    dP = torch.from_numpy(D["dPdrho"].reshape(-1)[:2].copy()).cuda()
    base = torch.from_numpy(fb).cuda()
    full = _solve(base, dP, th0, h, 9, True)
    lean = _solve(base, dP, th0, h, 9, True, want_X=False, want_dX=False, want_matrix=False)
    assert torch.equal(full.lam[:9], lean.lam[:9])
    only_dX = _solve(base, dP, th0, h, 9, True, want_X=False, want_dX=True)          # X is then internal scratch
    assert torch.equal(only_dX.dX[:9], full.dX[:9]) and torch.all(only_dX.dX[9:] == 0)
    fl = full.flags.cpu().numpy()
    assert np.all(fl[:9] == 0) and np.all(fl[9:] == 2)
    assert torch.isnan(full.lam[9:]).all() and torch.all(full.X[9:] == 0)


def test_scan_kernel_moves_matching_row(cuda_lib):
    """s-alpha lines with theta0 spread over [0, 20]: the 32 lanes of a warp have their eigenfunction peaks up to 600 rows
    apart, so no single matching row suits all of them -- the low-quality fallback (matching row moved, open solves
    re-converged) has to deliver every solve to full accuracy."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    from oracle import ballooning_oracle as bo
    theta = np.linspace(-10 * np.pi, 10 * np.pi, 2049)
    h = engine.grid_spacing(theta)
    cases = [(0.8, 0.8), (1.2, 0.4), (0.4, 0.6)]
    t0 = np.linspace(0.0, 20.0, 40)
    bases, dPs = zip(*[s_alpha_base(s, a, theta) for s, a in cases])
    base = torch.from_numpy(np.array(bases)).cuda()
    dP = torch.from_numpy(np.array(dPs)).cuda()
    th0 = torch.from_numpy(np.tile(t0, len(cases))).cuda()
    new = _solve(base, dP, th0, h, len(t0), True)
    old = _solve(base, dP, th0, h, len(t0), False)
    assert np.all(new.flags.cpu().numpy() == 0) and np.all(old.flags.cpu().numpy() == 0)
    np.testing.assert_allclose(new.lam.cpu().numpy(), old.lam.cpu().numpy(), rtol=LAM_RTOL, atol=0)
    np.testing.assert_allclose(new.X.cpu().numpy(), old.X.cpu().numpy(), rtol=0, atol=X_ATOL)
    assert np.ptp(np.argmax(new.X.cpu().numpy(), axis=1)) > 400          # the peaks really are far apart
    lam = new.lam.cpu().numpy()
    for s in (0, 17, 39, 40 + 25, 80 + 39):
        i, t = divmod(s, len(t0))
        b = bases[i]
        gam, X, *_ = bo.gamma_ball_full(dPs[i], theta, b[0], b[1], b[2] + t0[t] * b[3], b[4] + 2 * t0[t] * b[5] + t0[t] ** 2 * b[6],
                                        method="lambda_max")
        assert abs(lam[s] - gam) <= LAM_RTOL * abs(gam)
        np.testing.assert_allclose(new.X[s].cpu().numpy(), sign_normalise(X), rtol=0, atol=X_ATOL)


def test_scan_kernel_ineligible_batches_use_team_kernel(cuda_lib, golden):
    """Even N, fewer than four theta0, caller warm starts: not handled by the lane kernel -- the dispatch must fall back
    to the team kernel (same results either way)."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    D = golden("synthetic_d3d")
    theta = D["theta"][:-1]                                   # 1024 points: even
    h = engine.grid_spacing(theta)
    fb = fixture_base(D).reshape(-1, 8, len(D["theta"]))[:, :, :-1].copy()
    th0 = torch.from_numpy(np.tile(np.linspace(0, 1, 6), fb.shape[0])).cuda()
    a = _solve(torch.from_numpy(fb).cuda(), torch.from_numpy(D["dPdrho"].reshape(-1)).cuda(), th0, h, 6, True)
    b = _solve(torch.from_numpy(fb).cuda(), torch.from_numpy(D["dPdrho"].reshape(-1)).cuda(), th0, h, 6, False)
    assert torch.equal(a.lam, b.lam) and torch.equal(a.X, b.X)


@pytest.mark.parametrize("n", [65, 129, 257, 969])
def test_scan_kernel_small_and_odd_grids(cuda_lib, n):
    """Grids with 0, 1, 2 coarse levels and one whose coarse levels have an even number of points (969 = 8 * 121 + 1)."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    theta = np.linspace(-2 * np.pi, 2 * np.pi, n)
    h = engine.grid_spacing(theta)
    cases = [(0.8, 0.9), (1.1, 0.5)]
    bases, dPs = zip(*[s_alpha_base(s, a, theta) for s, a in cases])
    t0 = np.linspace(0.0, 1.2, 33)                        # two groups of lanes, the second with one active lane
    base, dP = torch.from_numpy(np.array(bases)).cuda(), torch.from_numpy(np.array(dPs)).cuda()
    th0 = torch.from_numpy(np.tile(t0, len(cases))).cuda()
    new = _solve(base, dP, th0, h, len(t0), True)
    old = _solve(base, dP, th0, h, len(t0), False)
    assert np.all(new.flags.cpu().numpy() == 0)
    np.testing.assert_allclose(new.lam.cpu().numpy(), old.lam.cpu().numpy(), rtol=LAM_RTOL, atol=0)
    np.testing.assert_allclose(new.X.cpu().numpy(), old.X.cpu().numpy(), rtol=0, atol=X_ATOL)
    np.testing.assert_allclose(new.dX.cpu().numpy(), old.dX.cpu().numpy(), rtol=0, atol=10 * X_ATOL * max(1.0, float(old.dX.abs().max())))


def test_scan_kernel_chunked_workspace(cuda_lib, golden):
    """IBS_SCAN_WS_MB bounds the coefficient workspace: the lines are then processed in chunks (here 2 lines per chunk),
    bit-identical to one launch."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    D = golden("synthetic_ncsx")
    theta = D["theta"]
    h = engine.grid_spacing(theta)
    fb = fixture_base(D)
    ns, na = fb.shape[:2]
    base, dP = torch.from_numpy(fb).cuda(), torch.from_numpy(D["dPdrho"]).cuda()
    th0 = torch.from_numpy(np.tile(np.linspace(0.0, 1.4, 9), ns * na)).cuda()
    sigma = torch.linspace(-1.0, 1.0, th0.numel(), dtype=torch.float64)
    one = _solve(base, dP, th0, h, 9, True, sigma=sigma)
    os.environ["IBS_SCAN_WS_MB"] = "1"
    try:
        many = _solve(base, dP, th0, h, 9, True, sigma=sigma)
    finally:
        os.environ.pop("IBS_SCAN_WS_MB", None)
    assert torch.equal(one.lam, many.lam) and torch.equal(one.X, many.X) and torch.equal(one.dX, many.dX)
    assert torch.equal(one.info, many.info) and torch.equal(one.lam_matrix, many.lam_matrix)


def test_lane_per_chain_warm_start_is_deterministic_and_changes_nothing(cuda_lib, monkeypatch):
    """The lane-per-chain kernel deals the lines in column order and warm-starts every line of rounds >= 1 from the previous
    line (ordered wait on its record, so the outcome does not depend on timing).  On a batch large enough for several rounds
    (20 D3D-like equilibria = 2560 lines x 64 theta0): two runs are bit-identical, the warm-started results equal the
    cold-started ones (IBS_SCAN_WARM=0) to rounding, the fused arg-max agrees, and the solver needs fewer passes."""
    import sys
    import torch
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
    import bench
    from ideal_ballooning_solver_b200 import engine
    st, alpha, theta0, theta = bench.build_tables("d3d", 20, seed0=100)
    dt = engine.DeviceTables.from_host(st)
    geo = engine.geometry_batch(dt, torch.from_numpy(alpha).cuda(), torch.from_numpy(theta).cuda())
    nt = theta0.size
    th0 = torch.from_numpy(theta0).cuda().repeat(st.ns)
    h = engine.grid_spacing(theta)

    def run():
        sol, best, sig = engine.scan_solve_argmax(geo.base, geo.dPdrho, th0, h, nt, 1, want_X=True)
        torch.cuda.synchronize()
        return sol, best, sig

    monkeypatch.setenv("IBS_SCAN_WARM", "1")
    a, best_a, sig_a = run()
    b, best_b, _ = run()
    assert torch.equal(a.lam, b.lam) and torch.equal(a.X, b.X) and torch.equal(best_a, best_b)
    monkeypatch.setenv("IBS_SCAN_WARM", "0")
    c, best_c, sig_c = run()
    assert int((a.info >> 16).max().item()) == 0 and int((c.info >> 16).max().item()) == 0
    scale = c.lam.abs().clamp_min(1e-3 * float(c.lam.abs().max().item()))
    assert float(((a.lam - c.lam).abs() / scale).max().item()) < 1e-11
    assert float((a.X - c.X).abs().max().item()) < 1e-9
    assert bool((a.X.max(dim=1).values == 1.0).all()) and bool((a.X >= 0).all())
    # the per-surface maxima: same winners unless two candidates tie to rounding
    same = best_a[:, 1] == best_c[:, 1]
    assert float(same.double().mean().item()) > 0.99
    assert float(((best_a[:, 0] - best_c[:, 0]).abs() / best_c[:, 0].abs().clamp_min(1e-6)).max().item()) < 1e-10
    it_w = float((a.info & 0xFFFF).double().mean().item()); it_c = float((c.info & 0xFFFF).double().mean().item())
    assert it_w < 0.95 * it_c, (it_w, it_c)           # (2560 lines = two rounds: half of them warm)


@pytest.mark.parametrize("scan2", ["1", "0"], ids=["scan2", "scan"])
def test_fused_argmax_guards_nan_and_tie(cuda_lib, monkeypatch, scan2):
    """The guarded per-surface arg-max fused into the lane kernels (ball_scan.py:279-295), on three surfaces of four s-alpha
    lines x 12 theta0 (N = 1025): a normal one; one with a NaN in one line's gds2, which gives (NaN, -2) and sigma0 = 0.05;
    one whose theta0 row repeats the theta0 of its maximum, so that two lanes of one item tie exactly and the first index
    wins.  Bit for bit against the stand-alone arg-max kernel on the returned lambda grid and against the oracle's rule."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    from oracle import ballooning_oracle as bo
    monkeypatch.setenv("IBS_SCAN", "1")
    monkeypatch.setenv("IBS_SCAN2", scan2)
    theta = np.linspace(-4 * np.pi, 4 * np.pi, 1025)
    h = engine.grid_spacing(theta)
    nsurf, lps, nth0 = 3, 4, 12
    cases = [(0.6 + 0.1 * q + 0.05 * l, 0.5 + 0.15 * l) for q in range(nsurf) for l in range(lps)]      # (shat, alpha) per line
    bases, dPs = zip(*[s_alpha_base(s, a, theta) for s, a in cases])
    base, dP = np.array(bases), np.array(dPs)
    base[lps + 1, 4, 300] = np.nan                                       # surface 1: a NaN in one line's gds2
    t0 = np.tile(np.linspace(0.0, 1.5, nth0), (nsurf * lps, 1))

    def run(t0):
        sol, best, sig = engine.scan_solve_argmax(torch.from_numpy(base).cuda(), torch.from_numpy(dP).cuda(),
                                                  torch.from_numpy(t0.ravel().copy()).cuda(), h, nth0, lps)
        val_r, idx_r, sig_r = engine.scan_argmax(sol.lam.reshape(nsurf, lps * nth0))
        lam, best, sig = sol.lam.cpu().numpy().reshape(nsurf, lps, nth0), best.cpu().numpy(), sig.cpu().numpy()
        assert np.array_equal(best[:, 0], val_r.cpu().numpy(), equal_nan=True)
        assert np.array_equal(best[:, 1], idx_r.cpu().numpy().astype(np.float64))
        assert np.array_equal(sig, sig_r.cpu().numpy())
        assert np.isnan(lam[1, 1]).all() and np.isnan(best[1, 0]) and best[1, 1] == -2.0 and sig[1] == 0.05
        for q in (0, 2):
            assert np.isfinite(lam[q]).all()
            ia, it, s0 = bo.argmax_with_guards(lam[q])
            assert best[q, 1] == ia * nth0 + it and best[q, 0] == lam[q, ia, it] and sig[q] == s0
        return lam, best

    lam, best = run(t0)
    la, it = divmod(int(best[2, 1]), nth0)
    j = it - 1 if it > 0 else it + 1                                     # another lane of the same item (nth0 <= 16)
    t0[2 * lps + la, j] = t0[2 * lps + la, it]
    lam, best = run(t0)
    assert lam[2, la, j] == lam[2, la, it] and np.count_nonzero(lam[2] == lam[2].max()) == 2
    assert best[2, 1] == la * nth0 + min(j, it)
