"""Reverse mode of K1 (``ibs_geometry_adjoint_scal`` through ``engine.geometry_adjoint``) against the long-double reference of
``geometry_ld``, and the per-point Hellmann-Feynman sensitivities (``ibs_adjoint_sensitivities``) against their closed form.

For one field line per surface and given cotangents (sg, sc, sf, Q) the kernel returns the gradient G of
    L(T) = sum_j [ sg_j g_j + sf_j f_j - dP sc_j chat_j ] - Q dPdrho
with respect to every Fourier table coefficient, the surface scalars (s, iota, iota', p', shat) and phiedge / Aminor_p.  L is
linear in the cotangents, so each channel (sg, sc, sf, Q) is driven alone with seeded random values, then all four together.
A direction delta is checked by
    err = |<G, delta> - dL_ld(delta)| / sum_q |delta_q G_q|
(for a scalar: |G_x - dL_ld| / sum_j |d Phi_j / dx|, Phi_j the per-point terms of the reference).  The directions:
  * per table row (6 ``mn`` rows, 7 Nyquist rows), two seeded "equalised" directions delta_q = +-r_q / max(|G_q|, floor),
    r_q in [0.5, 1]: every coefficient contributes about +-1, so one wrong coefficient moves err by ~1 / mnmax;
  * single coefficients at the edges of each mode set: (0, 0), the highest m, the highest +n and -n, the last Nyquist-only mode;
  * each scalar and global alone, and one mixed direction over everything;
  * lmns rows, iota and the mixed direction by full re-evaluation (Newton for theta_vmec included, independent of the kernel's
    implicit-function weight); every other direction by the exact linearity of the mode sums in the tables.

Derivatives that are zero identically (ZERO_ROWS: the Q channel sees no table coefficient and neither iota, iota' nor shat,
as (cvdrift - gbdrift) bmag^2 depends on s, p', phiedge and Aminor_p only; g and f do not depend on B_s, on the covariant
components of B or on p') are checked apart: |G| and |dL_ld| within ZERO_TOL of the reference's natural derivative size (the
size that moves the channel's terms by their own relative change at the step); measured <= 5e-15.  Any non-finite value fails.

Worst err per case measured on an NVIDIA B200 (1000 W power limit), over every channel and direction (rows / edge modes /
scalars and mixed / end to end):
  axisym_m20        5.8e-11 / 1.3e-14 / 5.8e-15          ntor16_nyq19      3.3e-13 / 1.4e-14 / 1.5e-14
  ntor5_nfp3        2.4e-12 / 7.4e-15 / 2.3e-14          ntor24_m18        2.5e-13 / 2.3e-14 / 2.2e-14
  ntor5_nfp3_phic   2.6e-12 / 1.4e-14 / 2.5e-14          ntor16_long       3.6e-12 / 1.2e-13 / 3.4e-14
  ntor11_nfp3       4.5e-13 / 2.3e-14 / 2.3e-14          synthetic_d3d     8.9e-11 / 1.7e-12 / 1.1e-14 / 5.4e-14
  ntor11_nfp3_phic  8.4e-13 / 2.0e-14 / 4.7e-14          ncsx_wout_op      1.1e-13 / 5.7e-14 / 1.1e-14 / 1.0e-14
ERR_BOUND is 10x the worst of each case, capped at 1e-10 (axisym_m20, synthetic_d3d).  The cases above ~1e-12 are set by the
equalised lmns directions, where the reference is the limit: its two Richardson estimates there differ by as much as err (up to
7e-11 on synthetic_d3d, 2.5e-11 on axisym_m20, 4e-12 on ntor5_nfp3 and ntor16_long), while every other direction of the same
cases is within ~2e-12.  An equalised lmns direction has its largest components on the coefficients with the smallest
gradient, so that the phases move far more than L does, and no step of the prescribed scheme is both free of truncation and
of rounding there.  Hence REF_SELF_GPU_LMNS.  The reference's own accuracy on the CPU self-checks below: its two Richardson
estimates agree to <= 1e-14 of the per-point scale (<= 3e-14 for the directions that move phi, where truncation at the
larger steps and rounding at the smaller ones cross at about 1.5e-14), the two routes agree to 1e-14, and L at T0 agrees with
the float64 oracle to 1e-13."""
import numpy as np
import pytest

from geometry_ld import Channel, L_ld, LineRef, dL_ld, linear_route_excluded, make_tables
from helpers import tables_from_fixture
from test_geometry_shapes_gpu import SHAPES

ROWS_MN = ("rmnc", "zmns", "lmns", "d_rmnc_d_s", "d_zmns_d_s", "d_lmns_d_s")
ROWS_NYQ = ("gmnc", "bmnc", "d_bmnc_d_s", "bsupvmnc", "bsubsmns", "bsubumnc", "bsubvmnc")
SIN_MN, SIN_NYQ = (1, 2, 4, 5), (4,)          # sine rows: the (0, 0) mode has no effect
SCALARS = ("s", "iota", "d_iota_d_s", "d_pressure_d_s", "shat", "phiedge", "Aminor_p")
CHANNELS = ("sg", "sc", "sf", "Q", "all")
FLOOR_REL = 1e-6           # equalised directions: |G_q| floored at FLOOR_REL x the row's largest |G_q| (per surface)
ERR_BOUND = {"axisym_m20": 1e-10, "ntor5_nfp3": 2.4e-11, "ntor5_nfp3_phic": 2.6e-11, "ntor11_nfp3": 4.5e-12,
             "ntor11_nfp3_phic": 8.3e-12, "ntor16_nyq19": 3.2e-12, "ntor24_m18": 2.5e-12, "ntor16_long": 3.6e-11, "synthetic_d3d": 1e-10,
             "ncsx_wout_op": 1.1e-12}
REF_SELF = 1e-14           # the reference's two Richardson estimates, relative to the per-point scale (CPU self-checks) ...
REF_SELF_PHI = 3e-14       # ... and for directions that move phi (iota, mixed): see the header
REF_SELF_GPU = 2e-12       # the same in the GPU comparisons, relative to the scale of err ...
REF_SELF_GPU_LMNS = 1e-10  # ... and for lmns directions (full re-evaluation of theta_vmec): see the header
ZERO_TOL = 1e-12           # identically zero derivatives: |G| and |dL_ld| relative to the reference's natural derivative size
MAX_REF_POINTS = 400       # the long line: cotangents on a seeded sample of this many points, Q = 0

# case -> (tables, ns, phi_center); synthetic shapes from test_geometry_shapes_gpu.SHAPES, golden fixtures by name
CASES = {
    "axisym_m20": ("axisym_m20", 3, 0.0),
    "ntor5_nfp3": ("ntor5_nfp3", 3, 0.0),
    "ntor5_nfp3_phic": ("ntor5_nfp3", 3, 0.7),
    "ntor11_nfp3": ("ntor11_nfp3", 3, 0.0),
    "ntor11_nfp3_phic": ("ntor11_nfp3", 3, -1.1),
    "ntor16_nyq19": ("ntor16_nyq19", 2, 0.0),
    "ntor24_m18": ("ntor24_m18", 2, 0.5),
    "ntor16_long": ("ntor16_long", 2, None),
    "synthetic_d3d": ("synthetic_d3d", 3, 0.0),
    "ncsx_wout_op": ("ncsx_wout_op", 2, 0.0),
}


# ---------------------------------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, name, golden):
        src, ns, phi_center = CASES[name]
        rng = np.random.default_rng(sum(map(ord, name)))
        if src in SHAPES:
            spec = SHAPES[src]
            self.st = make_tables(spec["mpol"], spec["ntor"], spec["nfp"], np.linspace(0.25, 0.9, ns), spec.get("extra_nyq"))
            self.theta = np.linspace(-spec["span"] * np.pi, spec["span"] * np.pi, spec["nl"])
            self.phi_center = spec.get("phi_center", 0.0) if phi_center is None else phi_center
        else:
            st = tables_from_fixture(golden(src))
            self.st = st.select(np.linspace(0, st.ns - 1, ns).round().astype(int))
            self.theta = np.linspace(-3 * np.pi, 3 * np.pi, 513)
            self.phi_center = phi_center
        self.name, self.ns, N = name, self.st.ns, self.theta.size
        self.alpha = rng.uniform(0.0, np.pi, self.ns)
        self.theta0 = np.array([0.0, 2.4, 0.8])[:self.ns]
        self.long = src == "ntor16_long"
        if self.long:
            self.cols = np.unique(np.concatenate([[0, N - 1], rng.choice(N, MAX_REF_POINTS - 2, replace=False)]))
        else:
            self.cols = np.arange(N)
        self.ref = LineRef(self.st, self.alpha, self.theta, self.theta0, self.phi_center, self.cols)
        q = self.ref.terms0[3].astype(np.float64)
        self.dP = -0.5 * q.mean(axis=-1)                  # dPdrho of the line (of the sample on a long line)
        self.channels = {}
        for k, nm in enumerate(CHANNELS):
            if nm == "Q" and self.long:
                continue
            r = np.random.default_rng([sum(map(ord, name)), k])
            vals = {}
            for c in ("sg", "sc", "sf"):
                v = np.zeros((self.ns, N))
                if nm in (c, "all"):
                    v[:, self.cols] = r.standard_normal((self.ns, self.cols.size))
                vals[c] = v
            Q = r.standard_normal(self.ns) if (nm in ("Q", "all") and not self.long) else np.zeros(self.ns)
            self.channels[nm] = Channel(vals["sg"], vals["sc"], vals["sf"], Q)
        self._G = {}

    def G(self, ch):
        """The kernel's gradient for channel ``ch``: (grad_mn, grad_nyq, grad_scal, grad_glob) as numpy arrays."""
        if ch not in self._G:
            from ideal_ballooning_solver_b200 import engine
            c = self.channels[ch]
            dt = engine.DeviceTables.from_host(self.st)
            out = engine.geometry_adjoint(dt, self.alpha, self.theta, self.theta0, self.dP, c.sg, c.sc, c.sf, c.Q,
                                          phi_center=self.phi_center, want_scalars=True)
            self._G[ch] = tuple(o.cpu().numpy() for o in out)
        return self._G[ch]


@pytest.fixture(scope="module")
def cases(golden):
    """Each case's tables, inputs and long-double reference line, built once per module on first use."""
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = Case(name, golden)
        return cache[name]
    return get


def edge_modes(xm, xn, mn_set=None):
    """Indices of the edge modes of one mode set: (0, 0), the highest m, the highest +n and -n and (Nyquist set, given the
    ``mn`` set) the last mode that is not in the ``mn`` set."""
    xm, xn = np.rint(xm).astype(int), np.rint(xn).astype(int)
    out = {"(0,0)": int(np.flatnonzero((xm == 0) & (xn == 0))[0]), "max m": int(np.flatnonzero(xm == xm.max())[0])}
    if xn.max() > 0:
        out["max +n"] = int(np.flatnonzero(xn == xn.max())[0])
        out["max -n"] = int(np.flatnonzero(xn == xn.min())[0])
    if mn_set is not None:
        known = set(zip(*(np.rint(a).astype(int) for a in mn_set)))
        only = [q for q in range(xm.size) if (xm[q], xn[q]) not in known]
        if only:
            out["last nyq-only"] = only[-1]
    return out


def _row_direction(st, which, row, vals):
    """Direction along one table row of every surface: ``vals (ns, nmodes)``."""
    tab = st.tab_mn if which == "mn" else st.tab_nyq
    d = np.zeros(tab.shape)
    d[:, row] = vals
    return {"tab_mn" if which == "mn" else "tab_nyq": d}


def _scalar_direction(st, x):
    if x in ("phiedge", "Aminor_p"):
        return {x: 1.0}
    d = np.zeros(st.scal.shape)
    d[:, SCALARS.index(x)] = 1.0
    return {"scal": d}


def _contract(G, direction):
    gmn, gnq, gsc, ggl = G
    out = np.zeros(gmn.shape[0])
    if "tab_mn" in direction:
        out += (gmn * direction["tab_mn"]).sum(axis=(1, 2))
    if "tab_nyq" in direction:
        out += (gnq * direction["tab_nyq"]).sum(axis=(1, 2))
    if "scal" in direction:
        out += (gsc * direction["scal"]).sum(axis=1)
    for k, col in (("phiedge", 0), ("Aminor_p", 1)):
        if k in direction:
            out += ggl[:, col] * direction[k]
    return out, _abs_terms(G, direction)


def _abs_terms(G, direction):
    gmn, gnq, gsc, ggl = G
    out = np.zeros(gmn.shape[0])
    if "tab_mn" in direction:
        out += np.abs(gmn * direction["tab_mn"]).sum(axis=(1, 2))
    if "tab_nyq" in direction:
        out += np.abs(gnq * direction["tab_nyq"]).sum(axis=(1, 2))
    if "scal" in direction:
        out += np.abs(gsc * direction["scal"]).sum(axis=1)
    for k, col in (("phiedge", 0), ("Aminor_p", 1)):
        if k in direction:
            out += np.abs(ggl[:, col] * direction[k])
    return out


def _route(direction):
    return "full" if linear_route_excluded(direction) else "linear"


# Derivatives that are zero identically (the channel's terms do not depend on the input): Q sees no table coefficient and
# neither iota, iota' nor shat, as (cvdrift - gbdrift) bmag^2 = -2 B_ref L_ref^2 sqrt(s) mu0 p' sgn / psi_e; g and f (channels
# sg, sf) do not depend on B_s or on the covariant components of B (they enter the drifts only), nor on p'.
ZERO_ROWS = {"Q": {("mn", r) for r in range(6)} | {("nyq", r) for r in range(7)} | {"iota", "d_iota_d_s", "shat"},
             "sg": {("nyq", 2), ("nyq", 4), ("nyq", 5), ("nyq", 6), "d_pressure_d_s"}}
ZERO_ROWS["sf"] = ZERO_ROWS["sg"]


def _ref_tol(which, row):
    return REF_SELF_GPU_LMNS if (which, row) == ("mn", 2) else REF_SELF_GPU


def _is_zero(ch, what):
    return what in ZERO_ROWS.get(ch, ())


class Tally:
    """Worst err (kernel against reference), worst reference self-agreement and worst |derivative| of the identically zero
    ones over the directions of one test; failures (and anything not finite) are collected and reported together."""

    def __init__(self, name):
        self.name, self.worst, self.worst_ref, self.worst_zero, self.bad = name, 0.0, 0.0, 0.0, []
        self.bound = ERR_BOUND[name]

    def add(self, what, got, scale, ref, zero=False, ref_tol=REF_SELF_GPU):
        """``scale``: sum_q |delta_q G_q| (0 for a scalar: the reference's per-point scale is used); ``zero``: the derivative
        is zero identically, so |got| and |d| are bounded by ZERO_TOL x the reference's natural derivative size instead."""
        d, d2, pscale, natural = (np.asarray(a, np.float64) for a in ref)
        got, scale = np.asarray(got, np.float64), np.asarray(scale, np.float64)
        if zero:
            e = np.maximum(np.abs(got), np.abs(d)) / natural
            self.worst_zero = float(np.max(np.concatenate([[self.worst_zero], e])))        # (np.max propagates NaN)
            if not np.all(e <= ZERO_TOL):                                                   # (False for NaN)
                self.bad.append((what, "zero", e, got, d))
            return
        scale = np.maximum(scale, pscale)
        both_zero = (got == 0) & (d == 0) & (d2 == 0)          # e.g. shat on a line with theta0 = 0 for sg, sc, sf: exact zeros
        pos = scale > 0
        err = np.where(pos, np.abs(got - d) / np.where(pos, scale, 1.0), np.where(both_zero, 0.0, np.inf))
        rerr = np.where(pos, np.abs(d - d2) / np.where(pos, scale, 1.0), np.where(both_zero, 0.0, np.inf))
        self.worst = float(np.max(np.concatenate([[self.worst], err])))
        self.worst_ref = float(np.max(np.concatenate([[self.worst_ref], rerr])))
        if not (np.all(err <= self.bound) and np.all(rerr <= ref_tol)):
            self.bad.append((what, err, rerr, got, d))

    def done(self, label):
        print("\n[adjoint-ld] %-18s %-8s worst err %.3e  reference self-agreement %.3e  zero derivatives %.3e"
              % (self.name, label, self.worst, self.worst_ref, self.worst_zero))
        assert not self.bad, (self.name, len(self.bad), self.bad[:5])
        assert np.isfinite(self.worst) and np.isfinite(self.worst_ref) and np.isfinite(self.worst_zero)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ---------------------------------------------------------------------------------------------------------------------
def _small_ref(phi_center=0.3, nl=65):
    st = make_tables(7, 5, 3, [0.3, 0.8])
    theta = np.linspace(-3 * np.pi, 3 * np.pi, nl)
    alpha, theta0 = np.array([0.2, 1.7]), np.array([0.0, 2.4])
    ref = LineRef(st, alpha, theta, theta0, phi_center)
    rng = np.random.default_rng(2)
    ch = Channel(*(rng.standard_normal((2, nl)) for _ in range(3)), rng.standard_normal(2))
    dP = -0.5 * ref.terms0[3].astype(np.float64).mean(axis=-1)
    return st, theta, alpha, theta0, ref, ch, dP


def _cpu_directions(st):
    rng = np.random.default_rng(4)
    d = {}
    for which, tab, rows in (("mn", st.tab_mn, range(6)), ("nyq", st.tab_nyq, range(7))):
        for row in rows:
            d["%s row %d" % (which, row)] = _row_direction(st, which, row, tab[:, row] * rng.uniform(-1, 1, tab[:, row].shape))
    for x in SCALARS:
        d[x] = _scalar_direction(st, x)
    d["mixed"] = {"tab_mn": st.tab_mn * rng.uniform(-1, 1, st.tab_mn.shape), "tab_nyq": st.tab_nyq * rng.uniform(-1, 1, st.tab_nyq.shape),
                  "scal": st.scal * rng.uniform(-1, 1, st.scal.shape), "phiedge": 0.3 * st.phiedge, "Aminor_p": -0.2 * st.Aminor_p}
    return d


def test_reference_L_agrees_with_float64_oracle():
    """L at T0 from the long-double reference (``L_ld``) and from the float64 oracle (``fieldlines`` -> ``gcf``,
    ``dpdrho_of``)."""
    from oracle import ballooning_oracle as bo
    st, theta, alpha, theta0, ref, ch, dP = _small_ref()
    phi = ref.contract(ref.terms0, dP, ch).astype(np.float64)
    L = L_ld(st, alpha, theta, theta0, dP, ch.sg, ch.sc, ch.sf, ch.Q, phi_center=0.3).astype(np.float64)
    assert np.array_equal(L, ref.L(dP, ch).astype(np.float64))
    for js in range(st.ns):
        fl = bo.fieldlines(st.select([js]), alpha[js:js + 1], theta, phi_center=0.3)
        cv, gd = bo.theta0_shift(fl, theta0[js])
        g, c, f = bo.gcf(dP[js], fl.bmag[0][0], fl.gradpar_theta_pest[0][0], cv, gd)
        want = np.sum(ch.sg[js] * g + ch.sc[js] * c + ch.sf[js] * f) - ch.Q[js] * bo.dpdrho_of(fl)
        assert abs(L[js] - want) <= 1e-13 * np.abs(phi[js]).sum(), (js, L[js], want)


def test_reference_richardson_estimates_agree():
    """The estimates from (h, h/2) and (2h, h) agree to REF_SELF of the per-point scale, on both routes, for a direction
    along every table row, every scalar, and a mixed one."""
    st, theta, alpha, theta0, ref, ch, dP = _small_ref()
    Q0 = Channel(ch.sg, ch.sc, ch.sf, np.zeros(2))
    for label, d in _cpu_directions(st).items():
        tol = REF_SELF_PHI if "scal" in d and np.any(d["scal"][:, 1] != 0) else REF_SELF
        for (dd, d2, scale, _) in ref.dL(d, dP, [ch, Q0], _route(d), check=True):
            dd, d2, scale = (a.astype(np.float64) for a in (dd, d2, scale))
            assert np.all(np.abs(dd - d2) <= tol * scale), (label, dd, d2, scale)


def test_reference_routes_agree():
    """Where both routes apply (``dL_ld`` with each) they agree to REF_SELF of the per-point scale; and the full route's
    evaluation by angle addition from the line at T0 agrees with evaluating the line from scratch, for a direction that moves
    theta_vmec and one that moves phi."""
    st, theta, alpha, theta0, ref, ch, dP = _small_ref(phi_center=-0.6)
    args = (st, alpha, theta, theta0, dP, ch.sg, ch.sc, ch.sf, ch.Q)
    for label, d in _cpu_directions(st).items():
        if linear_route_excluded(d):
            continue
        a, _, scale, _ = dL_ld(d, *args, phi_center=-0.6, route="linear")
        b, _, _, _ = dL_ld(d, *args, phi_center=-0.6, route="full")
        assert np.all(np.abs(a - b).astype(np.float64) <= REF_SELF * scale.astype(np.float64)), (label, a, b)
    # (from scratch, phi is formed from iota_t in long double: it differs from phi0 + dphi by phi0's float64 rounding)
    for label, tol in (("mn row 2", 1e-16), ("iota", 1e-13)):
        d = _cpu_directions(st)[label]
        h = ref.step(d, "full")
        fast, direct = ref.terms_full(d, h), ref.terms_full(d, h, direct=True)
        assert np.max(np.abs(fast - direct) / np.max(np.abs(direct), axis=-1, keepdims=True)) < tol, label


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernel's gradient against the reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_table_rows_equalised_directions(cuda_lib, cases, name):
    """Every table row, every channel: two equalised directions each (lmns by full re-evaluation)."""
    cs = cases(name)
    tally = Tally(name)
    for ch in cs.channels:
        G = cs.G(ch)
        rng = np.random.default_rng([sum(map(ord, name)), CHANNELS.index(ch)])
        for which, g_all, nrow, names in (("mn", G[0], 6, ROWS_MN), ("nyq", G[1], 7, ROWS_NYQ)):
            for row in range(nrow):
                g = g_all[:, row]
                floor = FLOOR_REL * np.max(np.abs(g), axis=-1, keepdims=True)
                floor[floor == 0] = 1.0           # a row this channel does not see (d_bmnc_d_s for sg, sf): G = 0 to check
                for k in range(2):
                    r = rng.uniform(0.5, 1.0, g.shape) * rng.choice([-1.0, 1.0], g.shape)
                    d = _row_direction(cs.st, which, row, r / np.maximum(np.abs(g), floor))
                    got, scale = _contract(G, d)
                    tally.add((ch, names[row], k), got, scale, cs.ref.dL(d, cs.dP, [cs.channels[ch]], _route(d), check=True)[0],
                              zero=_is_zero(ch, (which, row)), ref_tol=_ref_tol(which, row))
    tally.done("rows")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_table_edge_modes(cuda_lib, cases, name):
    """Single coefficients at the edges of each mode set, every row, every channel."""
    cs = cases(name)
    st = cs.st
    chans = list(cs.channels)
    Gs = [cs.G(ch) for ch in chans]
    tally = Tally(name)
    for which, xm, xn, nrow, sin_rows, names, mn_set in (("mn", st.xm, st.xn, 6, SIN_MN, ROWS_MN, None),
                                                         ("nyq", st.xm_nyq, st.xn_nyq, 7, SIN_NYQ, ROWS_NYQ, (st.xm, st.xn))):
        for label, q in edge_modes(xm, xn, mn_set).items():
            for row in range(nrow):
                if label == "(0,0)" and row in sin_rows:
                    continue
                vals = np.zeros((st.ns, xm.size))
                vals[:, q] = 1.0
                d = _row_direction(st, which, row, vals)
                refs = cs.ref.dL(d, cs.dP, [cs.channels[ch] for ch in chans], _route(d), check=True)
                for ch, G, ref in zip(chans, Gs, refs):
                    got, scale = _contract(G, d)
                    tally.add((ch, names[row], label), got, scale, ref, zero=_is_zero(ch, (which, row)), ref_tol=_ref_tol(which, row))
    tally.done("edges")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_scalars_and_mixed_direction(cuda_lib, cases, name):
    """Each of s, iota, iota', p', shat, phiedge, Aminor_p alone (iota by full re-evaluation, phi in long double), every
    channel; grad_scal[:, 5:] exactly 0; and one direction moving every table entry, scalar and global at once (full route)."""
    cs = cases(name)
    st = cs.st
    chans = list(cs.channels)
    Gs = [cs.G(ch) for ch in chans]
    tally = Tally(name)
    for G in Gs:
        assert np.all(G[2][:, 5:] == 0.0)
    for x in SCALARS:
        d = _scalar_direction(st, x)
        refs = cs.ref.dL(d, cs.dP, [cs.channels[ch] for ch in chans], _route(d), check=True)
        for ch, G, ref in zip(chans, Gs, refs):
            tally.add((ch, x), _contract(G, d)[0], 0.0, ref, zero=_is_zero(ch, x))
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    d = {"tab_mn": st.tab_mn * rng.uniform(-1, 1, st.tab_mn.shape), "tab_nyq": st.tab_nyq * rng.uniform(-1, 1, st.tab_nyq.shape),
         "scal": np.concatenate([st.scal[:, :5] * rng.uniform(-1, 1, (st.ns, 5)), np.zeros((st.ns, st.scal.shape[1] - 5))], axis=1),
         "phiedge": 0.3 * st.phiedge, "Aminor_p": -0.2 * st.Aminor_p}
    G = cs.G("all")
    got, scale = _contract(G, d)
    tally.add(("all", "mixed"), got, scale, cs.ref.dL(d, cs.dP, [cs.channels["all"]], "full", check=True)[0])
    tally.done("scalars")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synthetic_d3d", "ncsx_wout_op"])
def test_table_gradient_end_to_end(cuda_lib, golden, name):
    """``scan.table_gradient(..., scalars=True)`` with the genuine cotangents of the eigen-solve, formed as it forms them:
    ``adjoint_sensitivities``, then Q = sum sc c / (-dP).  One equalised direction per row and each scalar."""
    import torch
    from ideal_ballooning_solver_b200 import engine, scan
    st = tables_from_fixture(golden(name))
    theta = np.linspace(-3 * np.pi, 3 * np.pi, 513)
    rng = np.random.default_rng(5)
    a_star, t_star = rng.uniform(0.2, 2.5, st.ns), rng.uniform(0.0, 1.2, st.ns)
    t_star[0] = 2.2
    dt = engine.DeviceTables.from_host(st)
    tg = scan.table_gradient(dt, a_star, t_star, theta, scalars=True)
    a = torch.from_numpy(a_star[:, None].copy()).cuda()
    t0 = torch.from_numpy(t_star.copy()).cuda()
    geo = engine.geometry_batch(dt, a, theta)
    sol = engine.solve_base_batch(geo.base, geo.dPdrho, t0, engine.grid_spacing(theta), nth0=1, want_dX=True, want_matrix=False,
                                  want_gcf=True)
    sg, sc, sf = engine.adjoint_sensitivities(sol.lam, sol.X, sol.dX, sol.f)
    dP = geo.dPdrho.reshape(-1)
    Q = (sc * sol.c).sum(dim=1) / (-dP)
    ch = Channel(sg.cpu().numpy(), sc.cpu().numpy(), sf.cpu().numpy(), Q.cpu().numpy())
    dP = dP.cpu().numpy()
    G = (tg.grad_mn.cpu().numpy(), tg.grad_nyq.cpu().numpy(), tg.grad_scal.cpu().numpy(), tg.grad_glob.cpu().numpy())
    ref = LineRef(st, a_star, theta, t_star)
    tally = Tally(name)
    for which, g_all, nrow, names in (("mn", G[0], 6, ROWS_MN), ("nyq", G[1], 7, ROWS_NYQ)):
        for row in range(nrow):
            g = g_all[:, row]
            floor = FLOOR_REL * np.max(np.abs(g), axis=-1, keepdims=True)
            floor[floor == 0] = 1.0
            r = rng.uniform(0.5, 1.0, g.shape) * rng.choice([-1.0, 1.0], g.shape)
            d = _row_direction(st, which, row, r / np.maximum(np.abs(g), floor))
            got, scale = _contract(G, d)
            tally.add(names[row], got, scale, ref.dL(d, dP, [ch], _route(d), check=True)[0], ref_tol=_ref_tol(which, row))
    for x in SCALARS:
        d = _scalar_direction(st, x)
        tally.add(x, _contract(G, d)[0], 0.0, ref.dL(d, dP, [ch], _route(d), check=True)[0])
    tally.done("end-to-end")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: per-point sensitivities
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("N", [5, 6, 7, 64, 513, 1024])
def test_adjoint_sensitivities_closed_form(cuda_lib, N):
    """d lam / d g_j = -w_j dX_j^2 / Y1, d lam / d c_j = w_j X_j^2 / Y1, d lam / d f_j = -lam w_j X_j^2 / Y1 with Y1 =
    sum_j w_j f_j X_j^2 and w the weights of ``scipy.integrate.simpson`` (Cartwright's correction of the last interval at
    even N) (utils.py:1676-1680); and the per-point form contracted with perturbations equals ``adjoint_batch``."""
    import torch
    from scipy.integrate import simpson
    from ideal_ballooning_solver_b200 import engine
    rng = np.random.default_rng(N)
    ns = 3
    w = simpson(np.eye(N), axis=-1)
    X, dX = rng.standard_normal((ns, N)), rng.standard_normal((ns, N))
    f, lam = rng.uniform(0.5, 2.0, (ns, N)), rng.uniform(-1.0, 1.0, ns)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    sg, sc, sf = (t.cpu().numpy() for t in engine.adjoint_sensitivities(cu(lam), cu(X), cu(dX), cu(f)))
    Y1 = (w * f * X ** 2).sum(axis=-1, keepdims=True)
    for got, want in ((sg, -w * dX ** 2 / Y1), (sc, w * X ** 2 / Y1), (sf, -lam[:, None] * w * X ** 2 / Y1)):
        np.testing.assert_allclose(got, want, rtol=4e-15, atol=4e-16 * np.abs(want).max())
    npar = 4
    gp, cp, fp = (rng.standard_normal((ns, npar, N)) for _ in range(3))
    batch = engine.adjoint_batch(cu(lam), cu(X), cu(dX), cu(f), cu(gp), cu(cp), cu(fp)).cpu().numpy()
    per_point = (sg[:, None] * gp + sc[:, None] * cp + sf[:, None] * fp).sum(-1)
    scale = (np.abs(sg[:, None] * gp) + np.abs(sc[:, None] * cp) + np.abs(sf[:, None] * fp)).sum(-1)
    assert np.all(np.abs(batch - per_point) <= 1e-14 * scale), (batch, per_point)
