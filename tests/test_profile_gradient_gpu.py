"""Reverse mode of K1 with respect to the surface scalars (s, iota, iota', p', shat) and phiedge / Aminor_p
(``ibs_geometry_adjoint_scal``, ``scan.table_gradient(..., scalars=True)``): argument checks without a GPU; on the GPU
bit-identity of the table part with ``ibs_geometry_adjoint``, determinism, and the gradient against the finite-perturbation
Hellmann-Feynman form, against re-solved eigenvalues and for whole-equilibrium perturbations."""
import copy
import dataclasses

import numpy as np
import pytest

from helpers import tables_from_fixture

THETA = np.linspace(-3 * np.pi, 3 * np.pi, 513)
# (label, scal column or global name) of every input the scalar sweeps differentiate
SCALARS = (("s", 0), ("iota", 1), ("d_iota_d_s", 2), ("d_pressure_d_s", 3), ("shat", 4), ("phiedge", "phiedge"),
           ("Aminor_p", "Aminor_p"))


def _args(ns, ptr, grad_scal, grad_glob, phiedge=0.5, aminor_p=0.3):
    return (ptr, ptr, ptr, ptr, ptr, ptr, ptr, ns, 3, 4, phiedge, aminor_p, ptr, ptr, 9, 0.0, ptr, ptr, ptr, ptr, ptr, ptr,
            ptr, ptr, grad_scal, grad_glob, None)


def test_geometry_adjoint_scal_argument_errors_without_gpu():
    """Argument validation runs before any CUDA call and reports through ibs_last_error()."""
    from ideal_ballooning_solver_b200 import _lib, build
    build.build()
    lib = _lib.load()
    buf = np.zeros(64)
    p = buf.ctypes.data
    assert lib.ibs_geometry_adjoint_scal(*_args(0, None, None, None)) == 0
    assert lib.ibs_geometry_adjoint_scal(*_args(2, None, None, None)) == 1 and b"null" in lib.ibs_last_error()
    assert lib.ibs_geometry_adjoint_scal(*_args(2, p, None, p)) == 1 and b"null" in lib.ibs_last_error()
    assert lib.ibs_geometry_adjoint_scal(*_args(2, p, p, None)) == 1 and b"null" in lib.ibs_last_error()
    assert lib.ibs_geometry_adjoint_scal(*_args(2, p, p, p, aminor_p=0.0)) == 1 and b"Aminor_p" in lib.ibs_last_error()
    assert lib.ibs_geometry_adjoint_scal(*_args(2, p, p, p, aminor_p=-1.0)) == 1 and b"Aminor_p" in lib.ibs_last_error()
    assert lib.ibs_geometry_adjoint_scal(*_args(2, p, p, p, phiedge=0.0)) == 1 and b"phiedge" in lib.ibs_last_error()


# ---------------------------------------------------------------------------------------------------------------------
def _line(st, seed=5):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.2, 2.5, st.ns), rng.uniform(0.0, 1.2, st.ns)


def _perturbed(dt, which, delta):
    """Copy of the device tables with one scal column or one global moved by delta."""
    if isinstance(which, int):
        sc = dt.scal.clone()
        sc[:, which] += delta
        return dataclasses.replace(dt, scal=sc)
    return dataclasses.replace(dt, **{which: getattr(dt, which) + delta})


def _step(dt, which, rel):
    v = np.abs(dt.scal[:, which].cpu().numpy()).max() if isinstance(which, int) else abs(getattr(dt, which))
    return rel * v if v > 0 else rel


def _lam(dt, a_star, t_star):
    """lambda through the whole forward path (K1 + K2/K3) on the fixed lines (alpha*, theta0*)."""
    import torch
    from ideal_ballooning_solver_b200 import engine
    a = torch.from_numpy(np.asarray(a_star, dtype=np.float64)[:, None].copy()).cuda()
    t0 = torch.from_numpy(np.asarray(t_star, dtype=np.float64).copy()).cuda()
    geo = engine.geometry_batch(dt, a, THETA)
    return engine.solve_base_batch(geo.base, geo.dPdrho, t0, engine.grid_spacing(THETA), nth0=1, want_X=False, want_dX=False,
                                   want_matrix=False).lam.cpu().numpy()


@pytest.mark.gpu
def test_scalar_entry_point_tables_bit_identical_and_deterministic(cuda_lib, golden):
    import torch
    from ideal_ballooning_solver_b200 import engine
    st = tables_from_fixture(golden("synthetic_ncsx"))
    a_star, t_star = _line(st)
    dt = engine.DeviceTables.from_host(st)
    h = engine.grid_spacing(THETA)
    a = torch.from_numpy(a_star[:, None].copy()).cuda()
    t0 = torch.from_numpy(t_star.copy()).cuda()
    geo = engine.geometry_batch(dt, a, THETA)
    sol = engine.solve_base_batch(geo.base, geo.dPdrho, t0, h, nth0=1, want_dX=True, want_matrix=False, want_gcf=True)
    sg, sc, sf = engine.adjoint_sensitivities(sol.lam, sol.X, sol.dX, sol.f)
    dP = geo.dPdrho.reshape(-1)
    Q = (sc * sol.c).sum(dim=1) / (-dP)
    args = (dt, a.reshape(-1), THETA, t0, dP, sg, sc, sf, Q)
    gmn, gnq = engine.geometry_adjoint(*args)
    r1 = engine.geometry_adjoint(*args, want_scalars=True)
    r2 = engine.geometry_adjoint(*args, want_scalars=True)
    assert torch.equal(r1[0], gmn) and torch.equal(r1[1], gnq)
    assert r1[2].shape == (st.ns, 8) and r1[3].shape == (st.ns, 2)
    for x, y in zip(r1, r2):
        assert torch.equal(x, y)
    assert bool((r1[2][:, 5:] == 0).all())
    assert bool(torch.isfinite(r1[2]).all()) and bool(torch.isfinite(r1[3]).all())
    assert bool((r1[2][:, :5] != 0).all()) and bool((r1[3] != 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synthetic_ncsx", "synthetic_d3d", "ncsx_wout_op"])
def test_scalar_gradient_against_long_way(cuda_lib, golden, name):
    """Each scalar against the central difference of the finite-perturbation Hellmann-Feynman form (K1 re-run on the
    perturbed inputs, exact delta g, c, f, then the Hellmann-Feynman sums): isolates the adjoint of K1."""
    from ideal_ballooning_solver_b200 import engine, scan
    st = tables_from_fixture(golden(name))
    a_star, t_star = _line(st)
    dt0 = engine.DeviceTables.from_host(st)
    tg = scan.table_gradient(dt0, a_star, t_star, THETA, scalars=True)
    gsc, ggl = tg.grad_scal.cpu().numpy(), tg.grad_glob.cpu().numpy()
    sets, steps = [], []
    for _, which in SCALARS:
        step = _step(dt0, which, 1e-5)
        sets += [_perturbed(dt0, which, step), _perturbed(dt0, which, -step)]
        steps.append(step)
    hf = scan.hellmann_feynman_gamma(dt0, sets, a_star, t_star, THETA)
    np.testing.assert_allclose(tg.gamma, hf.gamma, rtol=1e-12)
    for k, (label, which) in enumerate(SCALARS):
        long_way = (hf.dgamma[2 * k] - hf.dgamma[2 * k + 1]) / (2.0 * steps[k])
        an = gsc[:, which] if isinstance(which, int) else ggl[:, 0 if which == "phiedge" else 1]
        np.testing.assert_allclose(an, long_way, rtol=2e-4, atol=1e-4 * np.abs(long_way).max() + 1e-13, err_msg=label)


@pytest.mark.gpu
def test_scalar_gradient_against_resolved_lambda(cuda_lib, golden):
    """Central differences of lambda itself through the whole forward path (the continuum Hellmann-Feynman formula is
    accurate to ~1e-3 on this grid)."""
    from ideal_ballooning_solver_b200 import engine, scan
    st = tables_from_fixture(golden("synthetic_ncsx"))
    a_star, t_star = _line(st)
    dt0 = engine.DeviceTables.from_host(st)
    tg = scan.table_gradient(dt0, a_star, t_star, THETA, scalars=True)
    gsc, ggl = tg.grad_scal.cpu().numpy(), tg.grad_glob.cpu().numpy()
    for label, which in (("iota", 1), ("d_pressure_d_s", 3), ("shat", 4), ("phiedge", "phiedge")):
        step = _step(dt0, which, 1e-5)
        fd = (_lam(_perturbed(dt0, which, step), a_star, t_star) - _lam(_perturbed(dt0, which, -step), a_star, t_star)) / (2 * step)
        an = gsc[:, which] if isinstance(which, int) else ggl[:, 0]
        np.testing.assert_allclose(an, fd, rtol=1e-2, atol=5e-3 * np.abs(fd).max() + 1e-12, err_msg=label)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["iota", "pressure", "phiedge", "all"])
def test_predict_with_scalars_for_equilibrium_perturbations(cuda_lib, case):
    """Perturbations of the whole equilibrium that move the profiles: TableGradient.predict with the scalar gradients
    against the finite-perturbation Hellmann-Feynman form and against re-solved eigenvalues.  Without the scalar gradients an
    iota-only perturbation is invisible to predict."""
    from ideal_ballooning_solver_b200 import engine, scan, synthetic, tables
    w = synthetic.make_equilibrium("ncsx", seed=11)
    s = np.linspace(0.55, 0.9, 6)
    st0 = tables.RadialSplines(w).evaluate(s)
    # iota moves the field line, phi = phi_c + (theta - alpha) / iota: at theta = 3 pi the phase of the n ~ 30 modes moves by
    # ~1e3 eps, so the second-order remainder of the finite perturbation is ~1e2 eps relative -- keep it well below 5e-4
    eps = 1.0e-6
    s_full = np.linspace(0.0, 1.0, w.ns)
    s_half = np.concatenate([[0.0], s_full[1:] - 0.5 * (s_full[1] - s_full[0])])
    wp = copy.copy(w)
    if case in ("iota", "all"):
        wp.iotas = w.iotas * (1.0 + eps * (1.0 + s_half))
    if case in ("pressure", "all"):
        wp.pres = w.pres * (1.0 + eps)
    if case in ("phiedge", "all"):
        wp.phi = w.phi * (1.0 + eps)
    if case == "all":
        rng = np.random.default_rng(7)
        wp.rmnc = w.rmnc * (1.0 + eps * rng.standard_normal(w.rmnc.shape[0])[:, None] * np.exp(-0.3 * np.arange(w.rmnc.shape[0]))[:, None])
    stp = tables.RadialSplines(wp).evaluate(s)
    a_star, t_star = _line(st0)
    dt0, dtp = engine.DeviceTables.from_host(st0), engine.DeviceTables.from_host(stp)
    tg = scan.table_gradient(dt0, a_star, t_star, THETA, scalars=True)
    pred = tg.predict(dt0, [dtp])[0]
    hf = scan.hellmann_feynman_gamma(dt0, [dtp], a_star, t_star, THETA)
    np.testing.assert_allclose(pred, hf.dgamma[0], rtol=5e-4, atol=1e-9 * np.abs(hf.dgamma).max())
    actual = _lam(dtp, a_star, t_star) - tg.gamma
    np.testing.assert_allclose(pred, actual, rtol=3e-3, atol=1e-12 * np.abs(tg.gamma).max() + 1e-14)
    if case == "iota":
        assert np.array_equal(stp.tab_mn, st0.tab_mn) and np.array_equal(stp.tab_nyq, st0.tab_nyq)
        pred_tables_only = scan.table_gradient(dt0, a_star, t_star, THETA).predict(dt0, [dtp])[0]
        assert np.all(pred_tables_only == 0.0)
        assert np.all(np.abs(actual) > 1e-3 * np.abs(pred).max())
