"""Extended-precision (long double, 64-bit mantissa) reference of K1's field-line geometry and of the scalar that its reverse
mode (``ibs_geometry_adjoint`` / ``ibs_geometry_adjoint_scal``) differentiates.  No tests live here.

The field line is split the way the kernels split it:
  * ``line_setup``: phi of every point, theta_vmec by Newton, and the trigonometric tables of both mode sets;
  * ``mode_sums``: the 19 mode sums.  At fixed theta_vmec and phi they are linear in the Fourier tables;
  * ``epilogue``: the pointwise algebra from the 19 sums and the surface constants to the eight base arrays.
``fieldlines_ld`` composes the three (``oracle.ballooning_oracle.fieldlines`` restated in long double).

The reverse mode returns the gradient of
    L(T) = sum_j [ sg_j g_j + sf_j f_j - dP sc_j chat_j ] - Q dPdrho,      dPdrho = -1/2 mean_j (cvdrift - gbdrift) bmag^2,
g = |gradpar| gd / bmag, chat = cv / (|gradpar| bmag), f = gd / (bmag^3 |gradpar|), cv and gd shifted by theta0, with dP held
fixed.  ``LineRef`` evaluates L and its directional derivatives along perturbations of the tables, the surface scalars and
the two globals: central differences at h and h / 2 in long double, combined by Richardson extrapolation, by one of two routes:
  * ``"full"``: everything re-evaluated at T0 + t delta, Newton for theta_vmec included.  Independent of the kernel's
    implicit-function weight; needed for directions that move theta_vmec (lmns) or phi (iota).
  * ``"linear"``: theta_vmec and phi stay put, the change of the sums is the sums of the direction itself (no step), and
    only the epilogue is differenced.  Valid for every direction that leaves lmns and iota alone; much cheaper."""
import dataclasses

import numpy as np

LD = np.longdouble
PI_LD = np.arccos(LD(-1))
MU0_LD = 4 * PI_LD * LD(10) ** -7
SUM_NAMES = ("R", "R_s", "R_t", "R_p", "Z_s", "Z_t", "Z_p", "L_s", "L_t", "L_p",
             "sqrtg", "B", "B_s", "B_t", "B_p", "Bsup_p", "Bsub_s", "Bsub_t", "Bsub_p")     # the kernels' S_* order
FULL_STEPS = ((3e-4, 1e-2), (1e-4, 1e-2), (3e-4, 1e-3))    # full route: (eps_rel, largest change of a phase m theta - n phi)
NSCAL_K1 = 5               # scal columns K1 reads: s, iota, iota', p', shat


# ---------------------------------------------------------------------------------------------------------------------
# synthetic tables
# ---------------------------------------------------------------------------------------------------------------------
def _append_nyq(st, n, frac=1e-4):
    """Append Nyquist modes (m, +-n nfp) for m = 0..3 with coefficients frac x the (m, 0) row."""
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


# ---------------------------------------------------------------------------------------------------------------------
# the field line in three parts
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class TablesLD:
    """Tables, surface scalars and globals in long double (T0 + t delta is formed without float64 rounding)."""
    tab_mn: np.ndarray
    tab_nyq: np.ndarray
    scal: np.ndarray
    phiedge: LD
    Aminor_p: LD
    xm: np.ndarray
    xn: np.ndarray
    xm_nyq: np.ndarray
    xn_nyq: np.ndarray

    @classmethod
    def of(cls, tab):
        if isinstance(tab, cls):
            return tab
        return cls(np.asarray(tab.tab_mn, LD), np.asarray(tab.tab_nyq, LD), np.asarray(tab.scal, LD), LD(tab.phiedge),
                   LD(tab.Aminor_p), np.asarray(tab.xm, np.float64), np.asarray(tab.xn, np.float64),
                   np.asarray(tab.xm_nyq, np.float64), np.asarray(tab.xn_nyq, np.float64))

    def moved(self, direction, t):
        """T + t direction (``direction``: dict with any of tab_mn, tab_nyq, scal, phiedge, Aminor_p)."""
        t = LD(t)
        get = lambda k, v: v + t * np.asarray(direction[k], LD) if k in direction else v
        return dataclasses.replace(self, tab_mn=get("tab_mn", self.tab_mn), tab_nyq=get("tab_nyq", self.tab_nyq),
                                   scal=get("scal", self.scal), phiedge=get("phiedge", self.phiedge),
                                   Aminor_p=get("Aminor_p", self.Aminor_p))


def line_phi(T, js, alpha, th_p, phi_center=0.0, phi_ld=False):
    """phi = phi_center + (theta_pest - alpha) / iota of the points (alpha (na,), th_p (nc,)) -> (phi64 or None, phi (LD)),
    both (na, nc).  By default formed in float64 exactly as K1 and the adjoint form it; ``phi_ld`` forms it in long double
    (a derivative in iota needs that: float64 phi would put 1e-16 / eps of noise into it)."""
    if phi_ld:
        phi = LD(phi_center) + (np.asarray(th_p, LD)[None, :] - np.asarray(alpha, LD)[:, None]) / T.scal[js, 1]
        return None, phi
    alpha = np.asarray(alpha, np.float64)
    phi64 = phi_center + (np.asarray(th_p, np.float64)[None, :] - alpha[:, None]) / np.float64(T.scal[js, 1])   # utils.py:373
    return phi64, phi64.astype(LD)


def theta_vmec(T, js, tp, phi, phi64=None):
    """theta_vmec + sum l sin(m theta_vmec - n phi) = theta_pest (utils.py:391-416) to long-double rounding; a float64 Newton
    supplies the start.  tp, phi: flat long-double arrays of the points."""
    xm, xn = T.xm.astype(LD), T.xn.astype(LD)
    lm = T.tab_mn[js, 2]
    lm64 = lm.astype(np.float64)
    p64 = phi.astype(np.float64) if phi64 is None else np.asarray(phi64, np.float64).ravel()
    tp64 = tp.astype(np.float64)
    th64 = tp64.copy()
    for _ in range(40):
        ang = T.xm[:, None] * th64[None] - T.xn[:, None] * p64[None]
        d = (th64 + lm64 @ np.sin(ang) - tp64) / (1 + (lm64 * T.xm) @ np.cos(ang))
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
    return th


@dataclasses.dataclass
class Trig:
    """cos / sin of m theta_vmec - n phi for both mode sets at the points of a line (flat)."""
    c: np.ndarray
    s: np.ndarray
    cq: np.ndarray
    sq: np.ndarray

    @classmethod
    def at(cls, T, th, phi):
        a = T.xm.astype(LD)[:, None] * th[None] - T.xn.astype(LD)[:, None] * phi[None]
        aq = T.xm_nyq.astype(LD)[:, None] * th[None] - T.xn_nyq.astype(LD)[:, None] * phi[None]
        return cls(np.cos(a), np.sin(a), np.cos(aq), np.sin(aq))


def mode_sums(tab_mn, tab_nyq, xm, xn, xmq, xnq, trig):
    """The 19 mode sums of one surface's rows (utils.py:420-468): ``tab_mn (6, mnmax)``, ``tab_nyq (7, mnmax_nyq)``.  Linear
    in the rows at fixed trig."""
    xm, xn, xmq, xnq = (np.asarray(a, LD) for a in (xm, xn, xmq, xnq))
    r, z, l, r_s, z_s, l_s = tab_mn
    R, R_s, Z_t, Z_p, L_t, L_p = np.stack([r, r_s, z * xm, -z * xn, l * xm, -l * xn]) @ trig.c
    R_t, R_p, Z_s, L_s = np.stack([-r * xm, r * xn, z_s, l_s]) @ trig.s
    g, b, b_s, bsupv, bsubs, bsubu, bsubv = tab_nyq
    sqrtg, B, B_s, Bsup_p, Bsub_t, Bsub_p = np.stack([g, b, b_s, bsupv, bsubu, bsubv]) @ trig.cq
    B_t, B_p, Bsub_s = np.stack([-b * xmq, b * xnq, bsubs]) @ trig.sq
    v = dict(R=R, R_s=R_s, R_t=R_t, R_p=R_p, Z_s=Z_s, Z_t=Z_t, Z_p=Z_p, L_s=L_s, L_t=L_t, L_p=L_p, sqrtg=sqrtg, B=B, B_s=B_s,
             B_t=B_t, B_p=B_p, Bsup_p=Bsup_p, Bsub_s=Bsub_s, Bsub_t=Bsub_t, Bsub_p=Bsub_p)
    return np.stack([v[k] for k in SUM_NAMES])


def epilogue(S, phi, scal_js, phiedge, Aminor_p, phi_center=0.0, phi_trig=None):
    """The eight base arrays from the 19 sums ``S (19, npt)`` and the surface constants (utils.py:474-720): Cartesian dual
    basis, grad psi, grad alpha, drifts, GS2 normalisations.  ``phi_trig``: (sin phi, cos phi, phi - phi_center) given
    instead of formed from ``phi``.  Returns a dict of long-double arrays."""
    R, R_s, R_t, R_p, Z_s, Z_t, Z_p, L_s, L_t, L_p, sqrtg, B, B_s, B_t, B_p, Bsup_p, Bsub_s, Bsub_t, Bsub_p = S
    s, iota, d_iota, dpds, shat = (LD(v) for v in scal_js[:5])
    psi_e = -LD(phiedge) / (2 * PI_LD)
    L_ref = LD(Aminor_p)
    B_ref = 2 * abs(psi_e) / (L_ref * L_ref)
    sgn = LD(np.sign(float(psi_e)))
    if phi_trig is None:
        sp, cp, phi_c = np.sin(phi), np.cos(phi), phi - LD(phi_center)
    else:
        sp, cp, phi_c = phi_trig
    X_t, X_p, X_s = R_t * cp, R_p * cp - R * sp, R_s * cp
    Y_t, Y_p, Y_s = R_t * sp, R_p * sp + R * cp, R_s * sp
    gs = [(Y_t * Z_p - Z_t * Y_p) / sqrtg, (Z_t * X_p - X_t * Z_p) / sqrtg, (X_t * Y_p - Y_t * X_p) / sqrtg]
    gt = [(Y_p * Z_s - Z_p * Y_s) / sqrtg, (Z_p * X_s - X_p * Z_s) / sqrtg, (X_p * Y_s - Y_p * X_s) / sqrtg]
    gp = [(Y_s * Z_t - Z_s * Y_t) / sqrtg, (Z_s * X_t - X_s * Z_t) / sqrtg, (X_s * Y_t - Y_s * X_t) / sqrtg]
    gpsi = [v * psi_e for v in gs]
    a_s = L_s - phi_c * d_iota
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
         "cvdrift0": -BxgB_gpsi * 2 * shat / (B * B * B * sqrt_s) * sgn}
    o["cvdrift"] = o["gbdrift"] - 2 * B_ref * L_ref * L_ref * sqrt_s * MU0_LD * dpds * sgn / (psi_e * B * B)
    return o


def line_setup(T, js, alpha, th_p, phi_center=0.0, phi_ld=False):
    """(phi, theta_vmec, Trig) of surface js at the points (alpha (na,), th_p (nc,)), all flat (na nc)."""
    phi64, phi = line_phi(T, js, alpha, th_p, phi_center, phi_ld)
    na = phi.shape[0]
    tp = np.broadcast_to(np.asarray(th_p, LD), (na, len(th_p))).ravel()
    phi = phi.ravel()
    th = theta_vmec(T, js, tp, phi, None if phi64 is None else phi64.ravel())
    return phi, th, Trig.at(T, th, phi)


def fieldlines_ld(tab, alpha, theta, phi_center=0.0, cols=None, phi_ld=False):
    """``oracle.ballooning_oracle.fieldlines`` (utils.py:161-720, hot subset) in long double.

    phi is formed in float64 exactly as K1 forms it, ``phi_center + (theta - alpha) / iota`` (``phi_ld``: in long double);
    from there on everything is long double.  theta_vmec is solved by Newton to the long-double rounding level (a float64
    Newton only supplies the start).  ``alpha`` is ``(nalpha,)`` or ``(ns, nalpha)`` (long double is kept with ``phi_ld``);
    ``cols`` picks the points of the line to evaluate (each point is independent).  Returns a dict of ``(ns, nalpha, ncols)`` long-double arrays: the eight base
    arrays and ``theta_vmec``."""
    from ideal_ballooning_solver_b200.engine import BASE_NAMES
    T = TablesLD.of(tab)
    theta = np.asarray(theta, dtype=np.float64)
    cols = np.arange(theta.size) if cols is None else np.asarray(cols)
    th_p = theta[cols]
    ns = T.tab_mn.shape[0]
    alpha = np.asarray(alpha, dtype=LD if phi_ld else np.float64)
    alpha2 = np.broadcast_to(alpha, (ns, alpha.shape[-1]))
    na, nc = alpha2.shape[1], th_p.size
    out = {k: np.empty((ns, na, nc), dtype=LD) for k in BASE_NAMES + ("theta_vmec",)}
    for js in range(ns):
        phi, th, trig = line_setup(T, js, alpha2[js], th_p, phi_center, phi_ld)
        S = mode_sums(T.tab_mn[js], T.tab_nyq[js], T.xm, T.xn, T.xm_nyq, T.xn_nyq, trig)
        o = epilogue(S, phi, T.scal[js], T.phiedge, T.Aminor_p, phi_center)
        o["theta_vmec"] = th
        for k, v in o.items():
            out[k][js] = v.reshape(na, nc)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the scalar the reverse mode differentiates, and its directional derivatives
# ---------------------------------------------------------------------------------------------------------------------
def point_terms(o, theta0):
    """(g, chat, f, q) of every point from the base arrays: q = (cvdrift - gbdrift) bmag^2, so dPdrho = -mean(q) / 2."""
    B, gp = o["bmag"], np.abs(o["gradpar_theta_pest"])
    th0 = LD(theta0)
    cv = o["cvdrift"] + th0 * o["cvdrift0"]
    gd = o["gds2"] + 2 * th0 * o["gds21"] + th0 * th0 * o["gds22"]
    return np.stack([gp * gd / B, cv / (gp * B), gd / (B * B * B * gp), (o["cvdrift"] - o["gbdrift"]) * B * B])


@dataclasses.dataclass
class Channel:
    """Cotangents of one evaluation of L: sg, sc, sf (ns, N), Q (ns,), with dP (ns,) held fixed."""
    sg: np.ndarray
    sc: np.ndarray
    sf: np.ndarray
    Q: np.ndarray


class LineRef:
    """One field line per surface (alpha_s, theta0_s, grid theta, phi_center) of tables T0, in long double.

    ``cols``: the points evaluated (default: those with a nonzero cotangent in any channel given later must be among them;
    with Q != 0 all N points are needed).  The line's phi, theta_vmec, trig tables and mode sums at T0 are computed once."""

    def __init__(self, tab, alpha, theta, theta0, phi_center=0.0, cols=None):
        self.T0 = TablesLD.of(tab)
        self.alpha = np.asarray(alpha, np.float64).reshape(-1)
        self.theta = np.asarray(theta, np.float64)
        self.theta0 = np.asarray(theta0, np.float64).reshape(-1)
        self.phi_center = float(phi_center)
        self.N = self.theta.size
        self.cols = np.arange(self.N) if cols is None else np.asarray(cols)
        self.ns = self.T0.tab_mn.shape[0]
        self.setup = [line_setup(self.T0, js, self.alpha[js:js + 1], self.theta[self.cols], self.phi_center)
                      for js in range(self.ns)]
        self.S0 = [mode_sums(self.T0.tab_mn[js], self.T0.tab_nyq[js], self.T0.xm, self.T0.xn, self.T0.xm_nyq, self.T0.xn_nyq,
                             self.setup[js][2]) for js in range(self.ns)]
        self.terms0 = self.terms_linear({}, 0)

        self._grouped = None

    # -- per-point terms (4, ns, ncols) at T0 + t delta ----------------------------------------------------------------
    def terms_full(self, direction, t, direct=False):
        """Full re-evaluation, Newton for theta_vmec included, by ``GroupedSums``: every phase is the phase at T0 plus a
        small change (m d theta_vmec - n d phi), so that nothing of the size of m theta - n phi (up to ~1e3) is rounded
        differently at different t.  ``direct``: the line evaluated from scratch instead (``line_setup``, phi in long double
        when the direction moves it), as a cross-check."""
        T = self.T0.moved(direction, t)
        dscal = np.asarray(direction.get("scal", np.zeros(T.scal.shape)), LD)
        moves_phi = bool(np.any(dscal[:, 1] != 0))
        if self._grouped is None and not direct:
            self._grouped = [GroupedSums(self.T0, js, *self.setup[js]) for js in range(self.ns)]
        out = []
        for js in range(self.ns):
            phi0 = self.setup[js][0]
            trig_phi = None
            if direct:
                phi, th, trig = line_setup(T, js, self.alpha[js:js + 1], self.theta[self.cols], self.phi_center, phi_ld=moves_phi)
                S = mode_sums(T.tab_mn[js], T.tab_nyq[js], T.xm, T.xn, T.xm_nyq, T.xn_nyq, trig)
            else:
                phi = phi0
                dmn = np.asarray(direction.get("tab_mn", np.zeros(T.tab_mn.shape)), LD)[js]
                dnq = np.asarray(direction.get("tab_nyq", np.zeros(T.tab_nyq.shape)), LD)[js]
                tp = self.theta[self.cols].astype(LD)
                if moves_phi:
                    # phi = phi0 + dphi, dphi = (theta - alpha) (1 / iota_t - 1 / iota_0), formed without phi0's rounding
                    i0, it = self.T0.scal[js, 1], T.scal[js, 1]
                    dphi = (tp - LD(self.alpha[js])) * (-LD(t) * dscal[js, 1]) / (it * i0)
                    sp0, cp0 = np.sin(phi0), np.cos(phi0)
                    cd, sd = np.cos(dphi), np.sin(dphi)
                    trig_phi = (sp0 * cd + cp0 * sd, cp0 * cd - sp0 * sd, (phi0 - LD(self.phi_center)) + dphi)
                    S = self._grouped[js].sums_at(dmn, dnq, t, tp, dphi=dphi, tabs=(T.tab_mn[js], T.tab_nyq[js]))
                else:
                    S = self._grouped[js].sums_at(dmn, dnq, t, tp)
            o = epilogue(S, phi, T.scal[js], T.phiedge, T.Aminor_p, self.phi_center, trig_phi)
            out.append(point_terms(o, self.theta0[js]))
        return np.stack(out, axis=1)

    def dsums(self, direction):
        """Change of the 19 sums per unit step along a direction that leaves theta_vmec and phi alone (exact: linear)."""
        T = self.T0
        zmn, znq = np.zeros(T.tab_mn.shape[1:], LD), np.zeros(T.tab_nyq.shape[1:], LD)
        dmn = np.asarray(direction.get("tab_mn", np.zeros(T.tab_mn.shape)), LD)
        dnq = np.asarray(direction.get("tab_nyq", np.zeros(T.tab_nyq.shape)), LD)
        out = []
        for js in range(self.ns):
            if not (dmn[js].any() or dnq[js].any()):
                out.append(None)
                continue
            out.append(mode_sums(dmn[js] if dmn[js].any() else zmn, dnq[js] if dnq[js].any() else znq, T.xm, T.xn,
                                 T.xm_nyq, T.xn_nyq, self.setup[js][2]))
        return out

    def terms_linear(self, direction, t, dS=None):
        assert not linear_route_excluded(direction), "the linear route needs theta_vmec and phi unchanged (no lmns, no iota)"
        T = self.T0.moved(direction, t)
        dS = self.dsums(direction) if dS is None else dS
        out = []
        for js in range(self.ns):
            S = self.S0[js] if dS[js] is None else self.S0[js] + LD(t) * dS[js]
            o = epilogue(S, self.setup[js][0], T.scal[js], T.phiedge, T.Aminor_p, self.phi_center)
            out.append(point_terms(o, self.theta0[js]))
        return np.stack(out, axis=1)

    # -- L ---------------------------------------------------------------------------------------------------------------
    def contract(self, terms, dP, ch):
        """Phi_j of every evaluated point (ns, ncols): sg g + sf f - dP sc chat + Q q / (2 N), so that L = sum_j Phi_j."""
        g, chat, f, q = terms
        c = self.cols
        dP = np.asarray(dP, LD).reshape(-1, 1)
        Q = np.asarray(ch.Q, LD).reshape(-1, 1)
        if np.any(Q != 0):
            assert self.cols.size == self.N, "Q != 0 needs every point of the line (dPdrho is a mean over all of them)"
        sg, sc, sf = (np.asarray(a, np.float64) for a in (ch.sg, ch.sc, ch.sf))
        mask = np.ones(self.N, bool)
        mask[c] = False
        assert not (sg[:, mask].any() or sc[:, mask].any() or sf[:, mask].any()), "nonzero cotangent on a point not evaluated"
        return (sg[:, c].astype(LD) * g + sf[:, c].astype(LD) * f - dP * sc[:, c].astype(LD) * chat
                + Q * q / (2 * LD(self.N)))

    def L(self, dP, ch, terms=None):
        return self.contract(self.terms0 if terms is None else terms, dP, ch).sum(axis=-1)

    def dL(self, direction, dP, channels, route="linear", h=None, check=False, eps_rel=3e-4):
        """Directional derivative of L along ``direction`` for each channel: a list of (d (ns,), d_2h (ns,) or None,
        scale (ns,), natural (ns,)) in long double.  d: Richardson (4 D(h/2) - D(h)) / 3 of the central differences; d_2h
        the same from 2h and h (``check``); scale: sum_j |d Phi_j| (the per-point derivatives, same extrapolation); natural:
        sum_j (|sg g| + |sf f| + |dP sc chat| + |Q q| / 2N) eps_rel / h, the size of a derivative that moves the channel's
        terms by their own relative change at the step (a derivative far below it is zero up to rounding).  h defaults to
        ``step(direction, route, eps_rel)``.  On the full route (h not given) the step is taken from FULL_STEPS, a few
        (eps_rel, phase limit) pairs: truncation dominates with the large ones on some lines, rounding with the small ones on
        others, and the pair whose two estimates agree best is used."""
        if route == "full" and h is None:
            best = None
            for e, ph in FULL_STEPS:
                res = self._dL(direction, dP, channels, route, self.step(direction, route, e, phase_rel=ph), True, e)
                worst = max(float(np.max(np.abs(d - d2) / np.maximum(sc, LD(1e-300)))) for d, d2, sc, _ in res)
                if best is None or worst < best[0]:
                    best = (worst, res)
            return best[1] if check else [(d, None, sc, nat) for d, _, sc, nat in best[1]]
        h = self.step(direction, route, eps_rel) if h is None else h
        return self._dL(direction, dP, channels, route, h, check, eps_rel)

    def _dL(self, direction, dP, channels, route, h, check, eps_rel):
        ev = self._evaluator(direction, route)
        ts = (h / 2, h, 2 * h) if check else (h / 2, h)
        diff = {t: (ev(t) - ev(-t)) for t in ts}
        out = []
        for ch in channels:
            D = {t: self.contract(diff[t], dP, ch) / (2 * LD(t)) for t in ts}     # per point (contract is linear in the terms)
            rich = (4 * D[h / 2] - D[h]) / 3
            rich2 = (4 * D[h] - D[2 * h]) / 3 if check else None
            nat = np.abs(self.contract(np.abs(self.terms0), np.abs(np.asarray(dP, LD)), Channel(*(np.abs(a) for a in (ch.sg, ch.sc, ch.sf, ch.Q)))))
            out.append((rich.sum(-1), None if rich2 is None else rich2.sum(-1), np.abs(rich).sum(-1), nat.sum(-1) * LD(eps_rel) / LD(h)))
        return out

    def _evaluator(self, direction, route):
        if route == "full":
            return lambda t: self.terms_full(direction, t)
        dS = self.dsums(direction)
        return lambda t: self.terms_linear(direction, t, dS)

    def step(self, direction, route, eps_rel=3e-4, ev=None, phase_rel=1e-2):
        """Step along the direction such that the per-point terms (g, chat, f, q) change by about eps_rel of their largest
        value on the line: a first step from a bound on the change of the mode sums, surface constants and (full route)
        phases m theta_vmec - n phi, then rescaled by the change that step actually makes."""
        T = self.T0
        nu = 0.0
        dS = self.dsums(direction)
        for js in range(self.ns):
            if dS[js] is not None:
                scale = np.maximum(np.max(np.abs(self.S0[js]), axis=1), LD(1e-300))
                nu = max(nu, float(np.max(np.max(np.abs(dS[js]), axis=1) / scale)))
        if "scal" in direction:
            d = np.asarray(direction["scal"], np.float64)[:, :NSCAL_K1]
            v = np.maximum(np.abs(T.scal[:, :NSCAL_K1].astype(np.float64)), 1e-3)
            nu = max(nu, float(np.max(np.abs(d) / v)))
        for k in ("phiedge", "Aminor_p"):
            if k in direction:
                nu = max(nu, abs(float(direction[k])) / abs(float(getattr(T, k))))
        nu_phase = 0.0
        if route == "full":
            mmax = float(np.max(T.xm)) + 1.0
            nmax = float(np.max(np.abs(np.concatenate([T.xn, T.xn_nyq])))) + 1.0
            if "tab_mn" in direction:
                dl = np.asarray(direction["tab_mn"], np.float64)[:, 2]
                nu_phase = max(nu_phase, float(np.max(np.abs(dl).sum(-1))) * mmax)
            if "scal" in direction:
                di = np.abs(np.asarray(direction["scal"], np.float64)[:, 1])
                dphi = np.max(np.abs(self.theta[self.cols][None, :] - self.alpha[:, None]), axis=1) / T.scal[:, 1].astype(np.float64) ** 2
                nu_phase = max(nu_phase, float(np.max(di * dphi)) * nmax)
        nu = max(nu, nu_phase)
        assert nu > 0, "zero direction"
        h0 = eps_rel / nu
        ev = self._evaluator(direction, route) if ev is None else ev
        rel = np.abs(ev(h0) - ev(-h0)) / (2 * np.max(np.abs(self.terms0), axis=-1, keepdims=True))
        rho = float(np.max(rel))
        h = h0 * min(eps_rel / rho, 1e6) if rho > 0 else h0
        return min(h, phase_rel / nu_phase) if nu_phase > 0 else h


class GroupedSums:
    """The 19 mode sums of one surface at ANY theta_vmec and phi near the line's, for any tables, by angle addition from the
    trig tables at (theta_vmec0, phi0): with d = theta_vmec - theta_vmec0,
        sum_q w_q cos(a_q + m_q d) = sum_m [ cos(m d) C_m(w) - sin(m d) S_m(w) ],   C_m(w) = sum_{q: m_q = m} w_q cos a_q,
    and the same for sin.  C_m, S_m are linear in the weights, so those of T0 + t delta are C_m(T0) + t C_m(delta).  A change
    dphi of phi first rotates a_q by -n_q dphi (then C_m, S_m are formed again).  Exact identities: the Newton solve for
    theta_vmec (in d, from 0) and the sums cost (distinct m) x points per evaluation, and only small angles are rounded."""
    ROWS_MN = (("r", 0, 0), ("rn", 0, 1), ("z", 1, 0), ("zn", 1, 1), ("l", 2, 0), ("ln", 2, 1), ("rs", 3, 0), ("zs", 4, 0), ("ls", 5, 0))
    ROWS_NYQ = (("g", 0, 0), ("b", 1, 0), ("bn", 1, 1), ("bs", 2, 0), ("bv", 3, 0), ("bsubs", 4, 0), ("bsubu", 5, 0), ("bsubv", 6, 0))

    def __init__(self, T, js, phi, th0, trig):
        self.th0 = th0
        self.sets = []
        for xm, xn, c, s, rows, key in ((T.xm, T.xn, trig.c, trig.s, self.ROWS_MN, "tab_mn"),
                                        (T.xm_nyq, T.xn_nyq, trig.cq, trig.sq, self.ROWS_NYQ, "tab_nyq")):
            perm = np.argsort(xm, kind="stable")
            um, starts = np.unique(xm[perm], return_index=True)
            un, ninv = np.unique(xn[perm], return_inverse=True)
            self.sets.append(dict(perm=perm, starts=starts, um=um.astype(LD), xn=np.asarray(xn, LD)[perm], c=c[perm], s=s[perm],
                                  rows=rows, key=key, un=un.astype(LD), ninv=ninv))
        self.base = self._grouped(T.tab_mn[js], T.tab_nyq[js])
        self._cache = {}

    def _grouped(self, tab_mn, tab_nyq, dphi=None):
        out = {}
        for st, tab in zip(self.sets, (tab_mn, tab_nyq)):
            c, s = st["c"], st["s"]
            if dphi is not None:                 # a - n dphi
                cu, su = np.cos(st["un"][:, None] * dphi[None]), np.sin(st["un"][:, None] * dphi[None])
                cn, sn = cu[st["ninv"]], su[st["ninv"]]
                c, s = c * cn + s * sn, s * cn - c * sn
            for name, row, npow in st["rows"]:
                w = np.asarray(tab[row], LD)[st["perm"]]
                if not w.any():
                    out[name] = None
                    continue
                if npow:
                    w = w * st["xn"]
                out[name] = (np.add.reduceat(w[:, None] * c, st["starts"], axis=0),
                             np.add.reduceat(w[:, None] * s, st["starts"], axis=0))
        return out

    def sums_at(self, dmn, dnq, t, theta_p, dphi=None, tabs=None):
        """The 19 sums at the theta_vmec of the tables T0 + t (dmn (6, mnmax), dnq (7, mnmax_nyq)) on this line; with
        ``dphi`` at phi0 + dphi, and ``tabs`` = (tab_mn, tab_nyq) of T0 + t delta."""
        if dphi is not None:
            G = self._grouped(*tabs, dphi=dphi)
        else:
            key = (dmn.tobytes(), dnq.tobytes())
            if key not in self._cache:
                self._cache = {key: self._grouped(dmn, dnq)}
            Gd, t = self._cache[key], LD(t)
            G = {k: (v if Gd[k] is None else (Gd[k] if v is None else (v[0] + t * Gd[k][0], v[1] + t * Gd[k][1])))
                 for k, v in self.base.items()}
        mn, nq = self.sets

        def cos_sum(st, g, d, mpow=0):           # sum_q w_q m^mpow cos(a_q + m d)
            if g is None:
                return np.zeros(d.shape, LD)
            um = st["um"][:, None]
            cm, sm = np.cos(um * d[None]), np.sin(um * d[None])
            return np.sum(um ** mpow * (cm * g[0] - sm * g[1]), axis=0)

        def sin_sum(st, g, d, mpow=0):
            if g is None:
                return np.zeros(d.shape, LD)
            um = st["um"][:, None]
            cm, sm = np.cos(um * d[None]), np.sin(um * d[None])
            return np.sum(um ** mpow * (cm * g[1] + sm * g[0]), axis=0)

        # theta_vmec + sum l sin(m theta_vmec - n phi) = theta_pest, Newton for d = theta_vmec - theta_vmec0 from 0: the
        # residual is r0 + d + sum, r0 = theta_vmec0 - theta_pest rounded once, the same at every t
        r0 = self.th0 - theta_p
        d = np.zeros_like(r0)
        extra = None
        for _ in range(30):
            dd = (r0 + d + sin_sum(mn, G["l"], d)) / (1 + cos_sum(mn, G["l"], d, 1))
            d = d - dd
            if extra is None and np.all(np.abs(dd) <= 1e-17):
                extra = 1                         # quadratic: one more correction reaches the rounding level
            elif extra is not None:
                break
        else:
            raise AssertionError("long-double Newton for theta_vmec did not converge")
        v = dict(R=cos_sum(mn, G["r"], d), R_s=cos_sum(mn, G["rs"], d), R_t=-sin_sum(mn, G["r"], d, 1),
                 R_p=sin_sum(mn, G["rn"], d), Z_s=sin_sum(mn, G["zs"], d), Z_t=cos_sum(mn, G["z"], d, 1),
                 Z_p=-cos_sum(mn, G["zn"], d), L_s=sin_sum(mn, G["ls"], d), L_t=cos_sum(mn, G["l"], d, 1),
                 L_p=-cos_sum(mn, G["ln"], d), sqrtg=cos_sum(nq, G["g"], d), B=cos_sum(nq, G["b"], d),
                 B_s=cos_sum(nq, G["bs"], d), B_t=-sin_sum(nq, G["b"], d, 1), B_p=sin_sum(nq, G["bn"], d),
                 Bsup_p=cos_sum(nq, G["bv"], d), Bsub_s=sin_sum(nq, G["bsubs"], d), Bsub_t=cos_sum(nq, G["bsubu"], d),
                 Bsub_p=cos_sum(nq, G["bsubv"], d))
        return np.stack([v[k] for k in SUM_NAMES])


def linear_route_excluded(direction):
    """True if the direction moves theta_vmec (an lmns row) or phi (iota)."""
    return (("tab_mn" in direction and np.any(np.asarray(direction["tab_mn"])[:, 2] != 0))
            or ("scal" in direction and np.any(np.asarray(direction["scal"])[:, 1] != 0)))


def L_ld(tables, alpha, theta, theta0, dP, sg, sc, sf, Q, phi_center=0.0, cols=None):
    """L of each surface (ns,) in long double (one field line per surface)."""
    ch = Channel(np.asarray(sg), np.asarray(sc), np.asarray(sf), np.asarray(Q, np.float64).reshape(-1))
    if cols is None and not np.any(ch.Q != 0):
        cols = np.flatnonzero(np.any((ch.sg != 0) | (ch.sc != 0) | (ch.sf != 0), axis=0))
    return LineRef(tables, alpha, theta, theta0, phi_center, cols).L(dP, ch)


def dL_ld(direction, tables, alpha, theta, theta0, dP, sg, sc, sf, Q, phi_center=0.0, cols=None, route=None, h=None,
          check=False):
    """Directional derivative of L (``LineRef.dL`` for one channel); ``route`` defaults to "full" for directions that move
    theta_vmec or phi and "linear" otherwise.  Returns (d, d_2h, scale, natural) per surface (``LineRef.dL``)."""
    ch = Channel(np.asarray(sg), np.asarray(sc), np.asarray(sf), np.asarray(Q, np.float64).reshape(-1))
    if cols is None and not np.any(ch.Q != 0):
        cols = np.flatnonzero(np.any((ch.sg != 0) | (ch.sc != 0) | (ch.sf != 0), axis=0))
    route = route or ("full" if linear_route_excluded(direction) else "linear")
    return LineRef(tables, alpha, theta, theta0, phi_center, cols).dL(direction, dP, [ch], route, h, check)[0]
