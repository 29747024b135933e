"""K1 (``ibs_geometry_batch``) on every code path of ``geometry_dispatch``, against an extended-precision field-line reference.

``geometry_dispatch`` picks the kernel from the toroidal width of the two mode sets (nt1 = max |xn| / nfp of the ``mn`` set,
nt2 the same for the Nyquist set): ``geometry_kernel<0,0>`` for axisymmetric tables, ``<6,8>``, ``<11,13>``, ``<16,18>``, and
``geometry3d_kernel`` above that (or with ``IBS_GEO3D=1``).  Each shape below is a synthetic equilibrium made to land on one of
them, at the widths on either side of every switch and at several field periods.  The reference, ``fieldlines_ld``, restates
``oracle.ballooning_oracle.fieldlines`` in long double (64-bit mantissa): it is ~1000x sharper than float64, so the bound on the
kernel is the kernel's own rounding and not the reference's.  ``engine.geometry_full`` is held to the same reference.

The argument checks of ``ibs_geometry_batch`` that run on the host before any CUDA call are tested without a GPU."""
import math
import re

import numpy as np
import pytest

LD = np.longdouble
PI_LD = np.arccos(LD(-1))
EPS = np.finfo(np.float64).eps

# Bounds, set from the worst case over all shapes measured on an NVIDIA B200 (1000 W power limit):
#   base arrays, relative to the row maximum: geometry_kernel<0,0> 4.5e-15, <6,8> 1.0e-14, <11,13> 8.6e-15, <16,18> 6.3e-14 (the
#   +-20 pi line; 1.7e-14 otherwise), geometry3d_kernel 2.1e-14, geometry_full 3.0e-14.
#   theta_vmec / (eps max(1, |theta_vmec|)): geometry_full 0.73, K1 13.7.  K1 stops Newton early once the error the last two
#   corrections predict (ad^3 / dprev^2) is below rounding; after the first two corrections from the start theta_pest that estimate
#   can be ~10x optimistic (seen in a float64 emulation of the iteration: with the early exit off, K1's rule gives 1.0 eps).
#   A few eps of theta_vmec move the base arrays by less than their bound.
BASE_RTOL = 2e-13          # each base array, relative to the maximum of its row (one surface, one alpha)
THETA_VMEC_EPS = 24        # theta_vmec within THETA_VMEC_EPS * eps * max(1, |theta_vmec|)

IBS_ERR_INVALID, IBS_ERR_UNSUPPORTED = 1, 3


# ---------------------------------------------------------------------------------------------------------------------
# extended-precision reference
# ---------------------------------------------------------------------------------------------------------------------
def fieldlines_ld(tab, alpha, theta, phi_center=0.0, cols=None):
    """``oracle.ballooning_oracle.fieldlines`` (utils.py:161-720, hot subset) in long double.

    phi is formed in float64 exactly as K1 forms it, ``phi_center + (theta - alpha) / iota``; from there on everything is long
    double.  theta_vmec is solved by Newton to the long-double rounding level (a float64 Newton only supplies the start).
    ``alpha`` is ``(nalpha,)`` or ``(ns, nalpha)``; ``cols`` picks the points of the line to evaluate (each point is
    independent).  Returns a dict of ``(ns, nalpha, ncols)`` long-double arrays: the eight base arrays and ``theta_vmec``."""
    from ideal_ballooning_solver_b200.engine import BASE_NAMES
    theta = np.asarray(theta, dtype=np.float64)
    cols = np.arange(theta.size) if cols is None else np.asarray(cols)
    th_p = theta[cols]
    ns = tab.tab_mn.shape[0]
    alpha = np.asarray(alpha, dtype=np.float64)
    alpha2 = np.broadcast_to(alpha, (ns, alpha.shape[-1]))
    na, nc = alpha2.shape[1], th_p.size
    xm, xn, xmq, xnq = (np.asarray(a, dtype=LD) for a in (tab.xm, tab.xn, tab.xm_nyq, tab.xn_nyq))
    xm64, xn64 = np.asarray(tab.xm, np.float64), np.asarray(tab.xn, np.float64)
    psi_e = -LD(tab.phiedge) / (2 * PI_LD)
    L_ref = LD(tab.Aminor_p)
    B_ref = 2 * abs(psi_e) / (L_ref * L_ref)
    sgn = LD(np.sign(float(psi_e)))
    MU0 = 4 * PI_LD * LD(10) ** -7
    out = {k: np.empty((ns, na, nc), dtype=LD) for k in BASE_NAMES + ("theta_vmec",)}
    for js in range(ns):
        sc = tab.scal[js]
        s, iota, d_iota, dpds, shat = (LD(v) for v in sc[:5])
        phi64 = phi_center + (th_p[None, :] - alpha2[js][:, None]) / sc[1]                   # utils.py:373, float64 as in K1
        phi, tp = phi64.astype(LD).ravel(), np.broadcast_to(th_p.astype(LD), (na, nc)).ravel()
        lm64 = tab.tab_mn[js, 2]
        lm = lm64.astype(LD)
        # theta_vmec + sum l sin(m theta_vmec - n phi) = theta_pest  (utils.py:391-416)
        th64 = tp.astype(np.float64)
        for _ in range(40):
            ang = xm64[:, None] * th64[None] - xn64[:, None] * phi64.ravel()[None]
            d = (th64 + lm64 @ np.sin(ang) - th_p[None, :].repeat(na, 0).ravel()) / (1 + (lm64 * xm64) @ np.cos(ang))
            th64 = th64 - d
            if np.max(np.abs(d)) < 1e-13:
                break
        th = th64.astype(LD)
        for _ in range(8):
            ang = xm[:, None] * th[None] - xn[:, None] * phi[None]
            d = (th + lm @ np.sin(ang) - tp) / (1 + (lm * xm) @ np.cos(ang))
            th = th - d
            if np.all(np.abs(d) <= 1e-18 * np.maximum(1, np.abs(th))):
                break
        else:
            raise AssertionError("long-double Newton for theta_vmec did not converge")
        # the 19 mode sums (utils.py:420-468)
        row = lambda k: tab.tab_mn[js, k].astype(LD)
        rowq = lambda k: tab.tab_nyq[js, k].astype(LD)
        r, z, l, r_s, z_s, l_s = (row(k) for k in range(6))
        ang = xm[:, None] * th[None] - xn[:, None] * phi[None]
        c, sn = np.cos(ang), np.sin(ang)
        R, R_s, Z_t, Z_p, L_t, L_p = np.stack([r, r_s, z * xm, -z * xn, l * xm, -l * xn]) @ c
        R_t, R_p, Z_s, L_s = np.stack([-r * xm, r * xn, z_s, l_s]) @ sn
        g, b, b_s, bsupv, bsubs, bsubu, bsubv = (rowq(k) for k in range(7))
        ang = xmq[:, None] * th[None] - xnq[:, None] * phi[None]
        c, sn = np.cos(ang), np.sin(ang)
        sqrtg, B, B_s, Bsup_p, Bsub_t, Bsub_p = np.stack([g, b, b_s, bsupv, bsubu, bsubv]) @ c
        B_t, B_p, Bsub_s = np.stack([-b * xmq, b * xnq, bsubs]) @ sn
        # Cartesian dual basis, grad psi, grad alpha, drifts, GS2 normalisations (utils.py:474-720)
        sp, cp = np.sin(phi), np.cos(phi)
        X_t, X_p, X_s = R_t * cp, R_p * cp - R * sp, R_s * cp
        Y_t, Y_p, Y_s = R_t * sp, R_p * sp + R * cp, R_s * sp
        gs = [(Y_t * Z_p - Z_t * Y_p) / sqrtg, (Z_t * X_p - X_t * Z_p) / sqrtg, (X_t * Y_p - Y_t * X_p) / sqrtg]
        gt = [(Y_p * Z_s - Z_p * Y_s) / sqrtg, (Z_p * X_s - X_p * Z_s) / sqrtg, (X_p * Y_s - Y_p * X_s) / sqrtg]
        gp = [(Y_s * Z_t - Z_s * Y_t) / sqrtg, (Z_s * X_t - X_s * Z_t) / sqrtg, (X_s * Y_t - Y_s * X_t) / sqrtg]
        gpsi = [v * psi_e for v in gs]
        a_s = L_s - (phi - LD(phi_center)) * d_iota
        ga = [a_s * gs[k] + ((1 + L_t) * gt[k] + (-iota + L_p) * gp[k]) for k in range(3)]
        BxgB_ga = (Bsub_s * B_t * (L_p - iota) + Bsub_t * B_p * a_s + Bsub_p * B_s * (1 + L_t) - Bsub_p * B_t * a_s
                   - Bsub_t * B_s * (L_p - iota) - Bsub_s * B_p * (1 + L_t)) / sqrtg
        ga_ga = ga[0] * ga[0] + ga[1] * ga[1] + ga[2] * ga[2]
        ga_gp = ga[0] * gpsi[0] + ga[1] * gpsi[1] + ga[2] * gpsi[2]
        gp_gp = gpsi[0] * gpsi[0] + gpsi[1] * gpsi[1] + gpsi[2] * gpsi[2]
        BxgB_gpsi = (Bsub_t * B_p - Bsub_p * B_t) / sqrtg * psi_e
        sqrt_s = np.sqrt(s)
        o = {"bmag": B / B_ref, "gradpar_theta_pest": L_ref * (iota * Bsup_p) / B, "gds2": ga_ga * L_ref * L_ref * s,
             "gds21": ga_gp * shat / B_ref, "gds22": gp_gp * shat * shat / (L_ref * L_ref * B_ref * B_ref * s),
             "gbdrift": -2 * B_ref * L_ref * L_ref * sqrt_s * BxgB_ga / (B * B * B) * sgn,
             "cvdrift0": -BxgB_gpsi * 2 * shat / (B * B * B * sqrt_s) * sgn, "theta_vmec": th}
        o["cvdrift"] = o["gbdrift"] - 2 * B_ref * L_ref * L_ref * sqrt_s * MU0 * dpds * sgn / (psi_e * B * B)
        for k, v in o.items():
            out[k][js] = v.reshape(na, nc)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# shapes: one synthetic equilibrium per code path and edge of geometry_dispatch
# ---------------------------------------------------------------------------------------------------------------------
K00, K68, K1113, K1618, K3D = "geometry_kernel<0,0>", "geometry_kernel<6,8>", "geometry_kernel<11,13>", "geometry_kernel<16,18>", "geometry3d_kernel"

# The synthetic Nyquist set has ntor + 2.  extra_nyq: |n| / nfp of Nyquist modes appended with small coefficients, so that nt2
# crosses a switch that nt1 does not reach.  span: the line is theta in shift + [-span pi, span pi]; three-point lines are shifted
# off theta = 0, +-pi, where the symmetric tables make some rows (cvdrift0) vanish and a row maximum is rounding noise.
SHAPES = {
    "axisym_m20":    dict(kernel=K00, mpol=20, ntor=0, nfp=1, nl=257, span=4),
    "axisym_nl3":    dict(kernel=K00, mpol=20, ntor=0, nfp=1, nl=3, span=1, shift=0.37),
    "ntor5_nfp3":    dict(kernel=K68, mpol=7, ntor=5, nfp=3, nl=1000, span=5),
    "ntor6_nfp2":    dict(kernel=K68, mpol=11, ntor=6, nfp=2, nl=257, span=3, per_surface_alpha=True),
    "ntor7_nfp5":    dict(kernel=K1113, mpol=11, ntor=7, nfp=5, nl=3, span=1, shift=0.37),
    "ntor11_nfp3":   dict(kernel=K1113, mpol=11, ntor=11, nfp=3, nl=257, span=3),
    "ntor12_nfp1":   dict(kernel=K1618, mpol=9, ntor=12, nfp=1, nl=1000, span=4),
    "ntor16_nfp2":   dict(kernel=K1618, mpol=13, ntor=16, nfp=2, nl=257, span=3, per_surface_alpha=True),
    "ntor17_nfp3":   dict(kernel=K3D, mpol=11, ntor=17, nfp=3, nl=1000, span=4),
    "ntor20_m12":    dict(kernel=K3D, mpol=12, ntor=20, nfp=5, nl=257, span=3),
    "ntor24_m18":    dict(kernel=K3D, mpol=18, ntor=24, nfp=2, nl=257, span=3, per_surface_alpha=True),
    "ntor6_nyq9":    dict(kernel=K1113, mpol=11, ntor=6, nfp=2, nl=257, span=3, extra_nyq=9),
    "ntor11_nyq14":  dict(kernel=K1618, mpol=11, ntor=11, nfp=3, nl=257, span=3, extra_nyq=14),
    "ntor16_nyq19":  dict(kernel=K3D, mpol=13, ntor=16, nfp=2, nl=257, span=3, extra_nyq=19),
    "ntor16_long":   dict(kernel=K1618, mpol=13, ntor=16, nfp=2, nl=4097, span=20, phi_center=0.4),
    "ntor24_long":   dict(kernel=K3D, mpol=18, ntor=24, nfp=2, nl=4097, span=20, phi_center=-1.3),
}
MAX_REF_POINTS = 400       # longer lines: the reference is evaluated on a seeded sample of this many points (and both ends)


def _append_nyq(st, n, frac=1e-4):
    """Append Nyquist modes (m, +-n nfp) for m = 0..3 with coefficients frac x the (m, 0) row."""
    import dataclasses
    xm, xn = [], []
    for m in range(4):
        for sgn in ((1,) if m == 0 else (1, -1)):
            xm.append(m)
            xn.append(sgn * n * st.nfp)
    src = [int(np.flatnonzero((st.xm_nyq == m) & (st.xn_nyq == 0))[0]) for m in xm]
    rng = np.random.default_rng(n)
    w = frac * rng.uniform(0.5, 1.0, len(xm))
    return dataclasses.replace(st, xm_nyq=np.concatenate([st.xm_nyq, xm]), xn_nyq=np.concatenate([st.xn_nyq, xn]),
                               tab_nyq=np.concatenate([st.tab_nyq, st.tab_nyq[:, :, src] * w], axis=2),
                               bsupumnc=np.concatenate([st.bsupumnc, st.bsupumnc[:, src] * w], axis=1))


def make_tables(mpol, ntor, nfp, s, extra_nyq=None, seed=1):
    """Surface tables of a synthetic equilibrium: a modified copy of the NCSX-shaped template (synthetic.py is unchanged)."""
    from ideal_ballooning_solver_b200 import synthetic, tables
    cfg = dict(synthetic.KINDS["ncsx"], mpol=mpol, ntor=ntor, nfp=nfp, ns=32)
    if ntor == 0:
        cfg["eps3d"] = 0.0
    kinds = dict(synthetic.KINDS, shape=cfg)
    orig = synthetic.KINDS
    synthetic.KINDS = kinds
    try:
        w = synthetic.make_equilibrium("shape", seed=seed)
    finally:
        synthetic.KINDS = orig
    st = tables.RadialSplines(w).evaluate(np.asarray(s, dtype=float))
    return _append_nyq(st, extra_nyq) if extra_nyq else st


def expected_kernel(st):
    """Python mirror of the kernel choice of ``geometry_dispatch`` (csrc/ibs_geometry.cu)."""
    xn_all = np.rint(np.concatenate([st.xn, st.xn_nyq])).astype(int)
    nfp = math.gcd(*[abs(int(v)) for v in xn_all]) or 1
    nt1 = int(np.max(np.abs(np.rint(st.xn)))) // nfp
    nt2 = int(np.max(np.abs(np.rint(st.xn_nyq)))) // nfp
    if nt1 == 0 and nt2 == 0:
        return K00
    if nt1 > 16 or nt2 > 18:
        return K3D
    if nt1 <= 6 and nt2 <= 8:
        return K68
    if nt1 <= 11 and nt2 <= 13:
        return K1113
    return K1618


class Shape:
    def __init__(self, name, spec):
        self.name, self.spec = name, spec
        ns = 2 if spec["ntor"] >= 20 else 3
        self.st = make_tables(spec["mpol"], spec["ntor"], spec["nfp"], np.linspace(0.25, 0.9, ns), spec.get("extra_nyq"))
        rng = np.random.default_rng(sum(map(ord, name)))
        self.theta = spec.get("shift", 0.0) + np.linspace(-spec["span"] * np.pi, spec["span"] * np.pi, spec["nl"])
        self.alpha = rng.uniform(0.0, np.pi, (ns, 3)) if spec.get("per_surface_alpha") else np.array([0.0, 0.9, 2.3])
        self.phi_center = spec.get("phi_center", 0.0)
        nl = spec["nl"]
        if nl > MAX_REF_POINTS:
            self.cols = np.unique(np.concatenate([[0, nl - 1], rng.choice(nl, MAX_REF_POINTS - 2, replace=False)]))
        else:
            self.cols = np.arange(nl)
        self._ref = None

    @property
    def ref(self):
        if self._ref is None:
            self._ref = fieldlines_ld(self.st, self.alpha, self.theta, self.phi_center, self.cols)
        return self._ref


@pytest.fixture(scope="module")
def shapes():
    """The tables and the long-double reference of each shape, built once per module on first use."""
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = Shape(name, SHAPES[name])
        return cache[name]
    return get


# ---------------------------------------------------------------------------------------------------------------------
# comparison helpers
# ---------------------------------------------------------------------------------------------------------------------
def run_k1(st, alpha, theta, phi_center=0.0):
    import torch
    from ideal_ballooning_solver_b200 import engine
    dt = engine.DeviceTables.from_host(st)
    geo = engine.geometry_batch(dt, torch.from_numpy(np.ascontiguousarray(alpha)).cuda(), torch.from_numpy(theta).cuda(),
                                phi_center=phi_center, want_theta_vmec=True, want_info=True)
    return (geo.base.cpu().numpy(), geo.theta_vmec.cpu().numpy(), geo.info.cpu().numpy(), geo.dPdrho.cpu().numpy())


def errors_against_ref(base, theta_vmec, ref, cols):
    """Per base array: max |got - ref| / (row max of |got|); theta_vmec: max |got - ref| / (eps max(1, |ref|))."""
    from ideal_ballooning_solver_b200.engine import BASE_NAMES
    err = {}
    for k, name in enumerate(BASE_NAMES):
        got = base[:, :, k, :]
        scale = np.max(np.abs(got), axis=-1)
        err[name] = float(np.max(np.abs(got[..., cols] - ref[name]).astype(np.float64) / scale[..., None]))
    r = ref["theta_vmec"]
    err["theta_vmec/eps"] = float(np.max((np.abs(theta_vmec[..., cols] - r) / np.maximum(1, np.abs(r))).astype(np.float64)) / EPS)
    return err


def assert_close_to_ref(err, what):
    bad = {k: v for k, v in err.items() if (v > THETA_VMEC_EPS if k == "theta_vmec/eps" else v > BASE_RTOL)}
    assert not bad, (what, bad)


def kernels_launched(fn):
    """Names of the CUDA kernels ``fn`` launches, as the profiler records them (whitespace removed)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {re.sub(r"\s+", "", e.name) for e in prof.events()}


def geometry_kernel_names(names):
    return sorted({m.group(0) for n in names for m in [re.search(r"geometry(3d)?_kernel(<\d+,\d+>)?", n)] if m})


# ---------------------------------------------------------------------------------------------------------------------
# host-side argument checks (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
def _batch_call(lib, xm, xn, xmq, xnq):
    """ibs_geometry_batch with host buffers: valid only for calls that fail in the host-side checks."""
    xm, xn, xmq, xnq = (np.ascontiguousarray(a, dtype=np.float64) for a in (xm, xn, xmq, xnq))
    buf = np.zeros(4096)
    p = buf.ctypes.data
    return lib.ibs_geometry_batch(p, p, p, xm.ctypes.data, xn.ctypes.data, xmq.ctypes.data, xnq.ctypes.data, 2, xm.size, xmq.size,
                                  0.5, 0.3, p, 3, 0, p, 9, 0.0, p, p, p, None, None)


@pytest.mark.parametrize("which,k,value", [("xm", 2, 1.5), ("xm", 1, -1.0), ("xn", 2, 3.5), ("xm_nyq", 3, 2.0 + 1e-6),
                                           ("xn_nyq", 1, -3.25)])
def test_non_integer_mode_numbers_rejected_without_gpu(which, k, value):
    """A fractional or negative m, or a fractional n, in either mode set is refused on the host before any CUDA call."""
    from ideal_ballooning_solver_b200 import _lib, build
    build.build()
    lib = _lib.load()
    modes = {"xm": np.array([0.0, 1.0, 1.0, 2.0]), "xn": np.array([0.0, -3.0, 3.0, 6.0])}
    modes["xm_nyq"], modes["xn_nyq"] = modes["xm"].copy(), modes["xn"].copy()
    modes[which][k] = value
    assert _batch_call(lib, modes["xm"], modes["xn"], modes["xm_nyq"], modes["xn_nyq"]) == IBS_ERR_INVALID
    assert b"non-integer mode numbers" in lib.ibs_last_error()


def test_mpol_too_large_for_3d_tables_rejected_without_gpu():
    """3-D tables hold 2 (mpol + 1) Newton coefficients per point in a fixed array: max xm >= 96 is refused on the host."""
    from ideal_ballooning_solver_b200 import _lib, build
    build.build()
    lib = _lib.load()
    xm, xn = np.array([0.0, 1.0, 96.0]), np.array([0.0, 2.0, -2.0])
    assert _batch_call(lib, xm, xn, xm, xn) == IBS_ERR_UNSUPPORTED
    assert b"mpol too large" in lib.ibs_last_error()


@pytest.mark.parametrize("mpol,ntor,nfp,per_surface", [(20, 0, 1, False), (7, 5, 3, True), (12, 20, 5, False)])
def test_reference_agrees_with_float64_oracle(mpol, ntor, nfp, per_surface):
    """The long-double reference and the float64 oracle (scipy secant for theta_vmec) are two statements of the same formulas:
    they agree to the oracle's rounding."""
    from oracle import ballooning_oracle as bo
    st = make_tables(mpol, ntor, nfp, [0.3, 0.8])
    theta = np.linspace(-3 * np.pi, 3 * np.pi, 65)
    alpha = np.array([[0.2, 1.7], [0.5, 2.9]]) if per_surface else np.array([0.2, 1.7])
    ref = fieldlines_ld(st, alpha, theta, phi_center=0.3)
    for js in range(st.ns):
        fl = bo.fieldlines(st.select([js]), alpha[js] if per_surface else alpha, theta, phi_center=0.3)
        r = {k: v[js:js + 1] for k, v in ref.items()}
        np.testing.assert_allclose(fl.theta_vmec, r["theta_vmec"].astype(float), rtol=0, atol=1e-13)
        for name in bo.HOT_FIELDS:
            got = getattr(fl, name)
            err = np.max(np.abs(got - r[name]).astype(float) / np.max(np.abs(got), axis=-1, keepdims=True))
            assert err < 1e-13, (name, err)


def test_dispatch_mirror_matches_shape_design():
    """Each shape's mode tables select the kernel the shape was made for (by the Python mirror of geometry_dispatch; the GPU
    tests check the mirror against the kernels the profiler records)."""
    import types
    from ideal_ballooning_solver_b200 import synthetic
    for name, spec in SHAPES.items():
        xm, xn = synthetic.vmec_mode_table(spec["mpol"] - 1, spec["ntor"], spec["nfp"])
        xmq, xnq = synthetic.vmec_mode_table(spec["mpol"] + 3, spec["ntor"] + 2 if spec["ntor"] else 0, spec["nfp"])
        if spec.get("extra_nyq"):
            xnq = np.concatenate([xnq, [-spec["extra_nyq"] * spec["nfp"]]])
        assert expected_kernel(types.SimpleNamespace(xm=xm, xn=xn, xm_nyq=xmq, xn_nyq=xnq)) == spec["kernel"], name


# ---------------------------------------------------------------------------------------------------------------------
# GPU: K1 and the full-output geometry against the reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SHAPES))
def test_k1_matches_extended_precision_reference(cuda_lib, shapes, monkeypatch, name):
    """The eight base arrays within BASE_RTOL of each row's maximum, theta_vmec within a few eps, Newton converged on every
    line, and dPdrho as the reference's formula gives it on the returned arrays.  Axisymmetric tables with the periodicity fold
    and without it."""
    from oracle import ballooning_oracle as bo
    from ideal_ballooning_solver_b200.engine import BASE_NAMES
    sh = shapes(name)
    for fold in (("1", "0") if sh.spec["ntor"] == 0 else ("1",)):
        monkeypatch.setenv("IBS_GEO_FOLD", fold)
        base, thv, info, dP = run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center)
        assert np.all(info >> 16 == 0) and np.all((info & 0xFFFF) <= 25), (name, fold, info)
        assert_close_to_ref(errors_against_ref(base, thv, sh.ref, sh.cols), (name, "fold=" + fold))
        fl = type("Fl", (), {n: base[:, :, k, :] for k, n in enumerate(BASE_NAMES)})
        want = np.array([[bo.dpdrho_of(fl, js, ja) for ja in range(base.shape[1])] for js in range(base.shape[0])])
        np.testing.assert_allclose(dP, want, rtol=1e-13, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SHAPES))
def test_geometry_full_matches_extended_precision_reference(cuda_lib, shapes, name):
    """``engine.geometry_full`` (mode 0: theta_pest grid) takes any mode list: the same shapes, the same reference, the same
    bounds."""
    from ideal_ballooning_solver_b200 import engine, reference_api
    from ideal_ballooning_solver_b200.engine import BASE_NAMES
    sh = shapes(name)
    idx = [reference_api.FULL_FIELDS.index(n) for n in BASE_NAMES + ("theta_vmec",)]
    rows = []
    for js in range(sh.st.ns):                    # (geometry_full takes one alpha list for all surfaces)
        al = sh.alpha[js] if sh.alpha.ndim == 2 else sh.alpha
        out, info = engine.geometry_full(sh.st.select([js]), al, sh.theta, mode=0, phi_center=sh.phi_center)
        info = info.cpu().numpy()
        assert np.all(info >> 16 == 0), (name, info)
        rows.append(out.cpu().numpy()[0][:, idx, :])
    got = np.stack(rows)
    assert_close_to_ref(errors_against_ref(got[:, :, :8], got[:, :, 8], sh.ref, sh.cols), (name, "geometry_full"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SHAPES))
def test_dispatch_runs_expected_kernel(cuda_lib, shapes, name):
    """The profiler sees exactly the geometry kernel instantiation the shape was made for."""
    sh = shapes(name)
    names = kernels_launched(lambda: run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center))
    assert geometry_kernel_names(names) == [sh.spec["kernel"]], (name, sorted(names))
    assert expected_kernel(sh.st) == sh.spec["kernel"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ntor5_nfp3", "ntor11_nfp3", "ntor16_nfp2"])
def test_forced_geometry3d_agrees_with_templated(cuda_lib, shapes, monkeypatch, name):
    """IBS_GEO3D=1 sends tables the templated kernels cover to geometry3d_kernel: same reference, and the two kernels agree
    with each other to rounding."""
    sh = shapes(name)
    base_t, thv_t, _, dP_t = run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center)
    monkeypatch.setenv("IBS_GEO3D", "1")
    names = kernels_launched(lambda: run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center))
    assert geometry_kernel_names(names) == [K3D]
    base, thv, info, dP = run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center)
    assert np.all(info >> 16 == 0)
    assert_close_to_ref(errors_against_ref(base, thv, sh.ref, sh.cols), (name, "IBS_GEO3D=1"))
    scale = np.max(np.abs(base_t), axis=-1, keepdims=True)
    assert np.max(np.abs(base - base_t) / scale) <= 2 * BASE_RTOL
    assert np.max(np.abs(thv - thv_t) / np.maximum(1, np.abs(thv_t))) <= 2 * THETA_VMEC_EPS * EPS
    np.testing.assert_allclose(dP, dP_t, rtol=4 * BASE_RTOL)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: batch composition and mode order
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["axisym_m20", "ntor6_nfp2", "ntor11_nfp3", "ntor16_nfp2", "ntor17_nfp3"])
def test_batch_composition_is_bit_identical(cuda_lib, name):
    """ns = 600 surfaces: each CTA takes several (surface, tile) work items and restages the tables where its range crosses into
    the next surface.  Every surface's output is bit-identical to the same surface in the batch in reversed order."""
    spec = SHAPES[name]
    st = make_tables(spec["mpol"], spec["ntor"], spec["nfp"], np.linspace(0.05, 0.95, 600), spec.get("extra_nyq"))
    theta = np.linspace(-3 * np.pi, 3 * np.pi, 257)
    alpha = np.array([0.0, 0.9, 2.3])
    fwd = run_k1(st, alpha, theta)
    rev = run_k1(st.select(np.arange(st.ns)[::-1]), alpha, theta)
    for a, b in zip(fwd, rev):
        assert np.array_equal(a, b[::-1])


def _permuted(st, perm_mn, perm_nyq):
    import dataclasses
    return dataclasses.replace(st, xm=st.xm[perm_mn], xn=st.xn[perm_mn], tab_mn=np.ascontiguousarray(st.tab_mn[:, :, perm_mn]),
                               xm_nyq=st.xm_nyq[perm_nyq], xn_nyq=st.xn_nyq[perm_nyq],
                               tab_nyq=np.ascontiguousarray(st.tab_nyq[:, :, perm_nyq]),
                               bsupumnc=np.ascontiguousarray(st.bsupumnc[:, perm_nyq]))


def _split_modes(st):
    """The same tables written differently: every m = 0, n > 0 mode as a (+n, -n) pair (half the coefficient each; the sine rows
    change sign at -n), and the (1, 0) and (1, nfp) modes of both sets split 3 : 5 across a duplicate entry."""
    import dataclasses
    SIN_MN, SIN_NYQ = [1, 2, 4, 5], [4]                  # zmns, lmns, d_zmns, d_lmns; bsubsmns

    def rewrite(xm, xn, tab, sin_rows):
        tab = tab.copy()
        pair = np.flatnonzero((xm == 0) & (xn > 0))
        tab[:, :, pair] *= 0.5
        neg = tab[:, :, pair].copy()
        neg[:, sin_rows] *= -1
        dup = np.concatenate([np.flatnonzero((xm == 1) & (xn == 0)), np.flatnonzero((xm == 1) & (xn == st.nfp))])
        extra = tab[:, :, dup] * 0.625
        tab[:, :, dup] *= 0.375
        return (np.concatenate([xm, xm[pair], xm[dup]]), np.concatenate([xn, -xn[pair], xn[dup]]),
                np.concatenate([tab, neg, extra], axis=2), pair, dup)

    xm, xn, tab_mn, _, _ = rewrite(st.xm, st.xn, st.tab_mn, SIN_MN)
    xmq, xnq, tab_nyq, pq, dq = rewrite(st.xm_nyq, st.xn_nyq, st.tab_nyq, SIN_NYQ)
    bu = st.bsupumnc.copy()
    bu[:, pq] *= 0.5
    extra = bu[:, dq] * 0.625
    bu[:, dq] *= 0.375
    bu = np.concatenate([bu, bu[:, pq], extra], axis=1)
    return dataclasses.replace(st, xm=xm, xn=xn, tab_mn=tab_mn, xm_nyq=xmq, xn_nyq=xnq, tab_nyq=tab_nyq, bsupumnc=bu)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["axisym_m20", "ntor6_nfp2", "ntor16_nfp2", "ntor17_nfp3"])
def test_mode_order_and_mode_splitting(cuda_lib, shapes, name):
    """A shuffled mode list gives bit-identical output (each packed cell receives the same additions); modes split across
    duplicate entries and m = 0 modes given as (+n, -n) pairs (both legal for the pack kernels) agree with the reference to
    rounding."""
    sh = shapes(name)
    ref_out = run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center)
    rng = np.random.default_rng(3)
    shuffled = _permuted(sh.st, rng.permutation(sh.st.xm.size), rng.permutation(sh.st.xm_nyq.size))
    for a, b in zip(ref_out, run_k1(shuffled, sh.alpha, sh.theta, sh.phi_center)):
        assert np.array_equal(a, b)
    split = _split_modes(sh.st)
    if sh.spec["ntor"] > 0:
        assert split.xm.size > sh.st.xm.size + 2 and np.any((split.xm == 0) & (split.xn < 0))
    assert expected_kernel(split) == sh.spec["kernel"]
    base, thv, info, _ = run_k1(split, sh.alpha, sh.theta, sh.phi_center)
    assert np.all(info >> 16 == 0)
    ref = fieldlines_ld(split, sh.alpha, sh.theta, sh.phi_center, sh.cols)
    assert_close_to_ref(errors_against_ref(base, thv, ref, sh.cols), (name, "split modes"))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: tables too large for shared memory
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ntor16_nfp2", "ntor17_nfp3"])
def test_tables_too_large_for_shared_memory(cuda_lib, shapes, name):
    """mpol 60 at these toroidal widths needs > 220 KB of shared memory per surface: IBS_ERR_UNSUPPORTED with its message, and
    the next normal call is unaffected."""
    import dataclasses
    from ideal_ballooning_solver_b200 import _lib
    sh = shapes(name)
    before = run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center)
    st = sh.st
    big = dataclasses.replace(st, xm=np.append(st.xm, 59.0), xn=np.append(st.xn, 0.0),
                              tab_mn=np.concatenate([st.tab_mn, np.zeros((st.ns, 6, 1))], axis=2),
                              xm_nyq=np.append(st.xm_nyq, 62.0), xn_nyq=np.append(st.xn_nyq, 0.0),
                              tab_nyq=np.concatenate([st.tab_nyq, np.zeros((st.ns, 7, 1))], axis=2))
    assert expected_kernel(big) == sh.spec["kernel"]
    with pytest.raises(_lib.IbsError, match=r"code 3\): Fourier tables of one surface do not fit in shared memory"):
        run_k1(big, sh.alpha, sh.theta, sh.phi_center)
    for a, b in zip(before, run_k1(sh.st, sh.alpha, sh.theta, sh.phi_center)):
        assert np.array_equal(a, b)
