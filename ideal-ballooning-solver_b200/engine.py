"""Batched tensor-in / tensor-out front end of the CUDA library (one process per GPU).

Every function takes and returns ``torch.float64`` CUDA tensors, launches on the current torch
stream and does not synchronise.  These are the calls the benchmarks, the scan driver and the
reference-signature facade (``reference_api.py``) are built on.
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import numpy as np
import torch

from . import _lib
from .tables import SurfaceTables

NBASE = 8
BASE_NAMES = ("bmag", "gradpar_theta_pest", "cvdrift", "cvdrift0", "gds2", "gds21", "gds22", "gbdrift")
FLAG_NOT_CONVERGED, FLAG_BAD_INPUT, FLAG_SIGMA_NOT_MAX = 1, 2, 4


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _f64(t, device, name):
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.asarray(t, dtype=np.float64))
    if t.dtype != torch.float64:
        raise TypeError(f"{name} must be float64")
    return t.to(device).contiguous()


def grid_spacing(theta) -> float:
    """``h`` exactly as ``gamma_ball_full`` forms it (``utils.py:1567-1575``)."""
    theta = np.asarray(theta, dtype=np.float64)
    tu = np.linspace(theta[0], theta[-1], len(theta))
    half = (tu[:-1] + tu[1:]) / 2
    return float(np.diff(half)[2]) if len(theta) > 3 else float(tu[1] - tu[0])


def fp64_peak_tflops(device=None, iters: int = 2000, reps: int = 5) -> float:
    """Measured FP64 FMA peak of the device in TFLOP/s (2 flops per FMA): the library's DFMA-chain probe timed with CUDA
    events, best of ``reps``.  Denominator of the FP64-pipe rooflines in ``bench.py``."""
    import ctypes
    _lib.require_cuda()
    lib = _lib.load()
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(dev):
        nsm = torch.cuda.get_device_properties(dev).multi_processor_count
        scratch = torch.empty(4 * nsm * 256, dtype=torch.float64, device=dev)
        nfma = ctypes.c_double(0.0)
        best = float("inf")
        for _ in range(reps + 1):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _lib.check(lib.ibs_fp64_probe(int(iters), scratch.data_ptr(), scratch.numel(), ctypes.byref(nfma), _stream()),
                       "ibs_fp64_probe")
            b.record()
            b.synchronize()
            best = min(best, a.elapsed_time(b))
    return 2.0 * nfma.value / (best * 1e-3) / 1e12


# ---------------------------------------------------------------------------------------------
@dataclasses.dataclass
class DeviceTables:
    """Per-surface Fourier tables resident in HBM (input contract of the geometry kernel)."""
    tab_mn: torch.Tensor     # (ns, 6, mnmax)
    tab_nyq: torch.Tensor    # (ns, 7, mnmax_nyq)
    scal: torch.Tensor       # (ns, 8)
    xm: np.ndarray
    xn: np.ndarray
    xm_nyq: np.ndarray
    xn_nyq: np.ndarray
    phiedge: float
    Aminor_p: float

    @classmethod
    def from_host(cls, st: SurfaceTables, device="cuda"):
        _lib.require_cuda()
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(device)
        c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        return cls(up(st.tab_mn), up(st.tab_nyq), up(st.scal), c(st.xm), c(st.xn), c(st.xm_nyq), c(st.xn_nyq),
                   float(st.phiedge), float(st.Aminor_p))

    @property
    def ns(self):
        return self.tab_mn.shape[0]


@dataclasses.dataclass
class Geometry:
    base: torch.Tensor                   # (ns, nalpha, 8, nl)
    dPdrho: torch.Tensor                 # (ns, nalpha)
    theta_vmec: Optional[torch.Tensor]   # (ns, nalpha, nl)
    info: Optional[torch.Tensor]         # (ns, nalpha) int32

    def field(self, name):
        return self.base[:, :, BASE_NAMES.index(name), :]


def geometry_batch(tables: DeviceTables, alpha, theta, phi_center: float = 0.0, want_theta_vmec: bool = False,
                   want_info: bool = False) -> Geometry:
    """K1: ``vmec_fieldlines`` for ``ns`` surfaces x ``nalpha`` lines x ``nl`` points
    (``utils.py:161-864``).  ``alpha`` is ``(nalpha,)`` (shared) or ``(ns, nalpha)`` (per surface)."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = tables.tab_mn.device
    alpha = _f64(alpha, dev, "alpha")
    theta = _f64(theta, dev, "theta")
    per_surface = alpha.dim() == 2
    if per_surface and alpha.shape[0] != tables.ns:
        raise ValueError("alpha must be (nalpha,) or (ns, nalpha)")
    ns, nalpha, nl = tables.ns, alpha.shape[-1], theta.numel()
    base = torch.empty((ns, nalpha, NBASE, nl), dtype=torch.float64, device=dev)
    dP = torch.empty((ns, nalpha), dtype=torch.float64, device=dev)
    thv = torch.empty((ns, nalpha, nl), dtype=torch.float64, device=dev) if want_theta_vmec else None
    info = torch.empty((ns, nalpha), dtype=torch.int32, device=dev) if want_info else None
    with torch.cuda.device(dev):
        rc = lib.ibs_geometry_batch(_ptr(tables.tab_mn), _ptr(tables.tab_nyq), _ptr(tables.scal),
                                    tables.xm.ctypes.data, tables.xn.ctypes.data, tables.xm_nyq.ctypes.data,
                                    tables.xn_nyq.ctypes.data, ns, len(tables.xm), len(tables.xm_nyq),
                                    tables.phiedge, tables.Aminor_p, _ptr(alpha), nalpha, int(per_surface),
                                    _ptr(theta), nl, float(phi_center), _ptr(base), _ptr(dP), _ptr(thv), _ptr(info),
                                    _stream())
    _lib.check(rc, "ibs_geometry_batch")
    return Geometry(base, dP, thv, info)


@dataclasses.dataclass
class GeometryTangent(Geometry):
    dbase: Optional[torch.Tensor] = None      # (ns, nalpha, 8, nl)  d base / d alpha at fixed theta_pest
    ddPdrho: Optional[torch.Tensor] = None    # (ns, nalpha)         d dPdrho / d alpha


def geometry_tangent_batch(tables: DeviceTables, alpha, theta, phi_center: float = 0.0, want_theta_vmec: bool = False,
                           want_info: bool = False) -> GeometryTangent:
    """K1 and its exact alpha-derivative (``ibs_geometry_tangent_batch``): the ``Geometry`` of ``geometry_batch`` (the same
    bits) plus ``dbase`` and ``ddPdrho``, the derivatives of the eight base arrays and of dPdrho with respect to the field-line
    label alpha at fixed theta_pest.  ``alpha`` is ``(nalpha,)`` (shared) or ``(ns, nalpha)`` (per surface)."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = tables.tab_mn.device
    alpha = _f64(alpha, dev, "alpha")
    theta = _f64(theta, dev, "theta")
    per_surface = alpha.dim() == 2
    if per_surface and alpha.shape[0] != tables.ns:
        raise ValueError("alpha must be (nalpha,) or (ns, nalpha)")
    ns, nalpha, nl = tables.ns, alpha.shape[-1], theta.numel()
    base = torch.empty((ns, nalpha, NBASE, nl), dtype=torch.float64, device=dev)
    dbase = torch.empty_like(base)
    dP = torch.empty((ns, nalpha), dtype=torch.float64, device=dev)
    ddP = torch.empty_like(dP)
    thv = torch.empty((ns, nalpha, nl), dtype=torch.float64, device=dev) if want_theta_vmec else None
    info = torch.empty((ns, nalpha), dtype=torch.int32, device=dev) if want_info else None
    with torch.cuda.device(dev):
        rc = lib.ibs_geometry_tangent_batch(_ptr(tables.tab_mn), _ptr(tables.tab_nyq), _ptr(tables.scal),
                                            tables.xm.ctypes.data, tables.xn.ctypes.data, tables.xm_nyq.ctypes.data,
                                            tables.xn_nyq.ctypes.data, ns, len(tables.xm), len(tables.xm_nyq),
                                            tables.phiedge, tables.Aminor_p, _ptr(alpha), nalpha, int(per_surface),
                                            _ptr(theta), nl, float(phi_center), _ptr(base), _ptr(dP), _ptr(dbase), _ptr(ddP),
                                            _ptr(thv), _ptr(info), _stream())
    _lib.check(rc, "ibs_geometry_tangent_batch")
    return GeometryTangent(base, dP, thv, info, dbase, ddP)


def geometry_full(st: SurfaceTables, alpha, grid, mode: int = 0, theta_shift: float = 0.0, zero_xn_nyq: bool = False,
                  phi_center: float = 0.0, device="cuda"):
    """Every per-point array of the reference's ``vmec_fieldlines`` / ``vmec_fieldlines_axisym`` Struct
    (``utils.py:723-864``, ``:872-1542``) through ``ibs_geometry_full`` (not a hot kernel).  ``mode`` 0: ``grid`` is
    theta_pest, 1: phi, 2: theta_vmec (no root solve).  Returns ``(out (ns, nalpha, NF, nl), info (ns, nalpha))``;
    field order = ``reference_api.FULL_FIELDS``."""
    _lib.require_cuda()
    lib = _lib.load()
    if st.bsupumnc is None:
        raise ValueError("the full-output geometry needs the bsupumnc table (SurfaceTables.bsupumnc)")
    dev = torch.device(device)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    tab_mn, tab_nyq, bsu, scal = up(st.tab_mn), up(st.tab_nyq), up(st.bsupumnc), up(st.scal)
    xm, xn, xmq, xnq = up(st.xm), up(st.xn), up(st.xm_nyq), up(st.xn_nyq)
    alpha, grid = up(np.atleast_1d(alpha)), up(np.atleast_1d(grid))
    ns, na, nl = st.ns, alpha.numel(), grid.numel()
    nf = lib.ibs_geometry_full_nfields()
    out = torch.empty((ns, na, nf, nl), dtype=torch.float64, device=dev)
    info = torch.empty((ns, na), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ibs_geometry_full(_ptr(tab_mn), _ptr(tab_nyq), _ptr(bsu), _ptr(scal), _ptr(xm), _ptr(xn), _ptr(xmq), _ptr(xnq),
                                   ns, xm.numel(), xmq.numel(), float(st.phiedge), float(st.Aminor_p), _ptr(alpha), na, _ptr(grid), nl,
                                   int(mode), float(theta_shift), int(bool(zero_xn_nyq)), float(phi_center), _ptr(out), _ptr(info),
                                   _stream())
    _lib.check(rc, "ibs_geometry_full")
    return out, info


# ---------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Solution:
    lam: torch.Tensor                      # (nsolve,) Simpson Rayleigh quotient = the reference's `gam`
    lam_matrix: Optional[torch.Tensor]     # (nsolve,) lambda_max of the discrete pencil
    X: Optional[torch.Tensor]              # (nsolve, N)
    dX: Optional[torch.Tensor]
    info: torch.Tensor                     # (nsolve,) int32: iterations | flags << 16
    g: Optional[torch.Tensor] = None
    c: Optional[torch.Tensor] = None
    f: Optional[torch.Tensor] = None

    @property
    def iterations(self):
        return self.info & 0xFFFF

    @property
    def flags(self):
        return self.info >> 16


def _alloc_out(n, N, dev, want_X, want_dX, want_matrix):
    lam = torch.empty((n,), dtype=torch.float64, device=dev)
    lm = torch.empty((n,), dtype=torch.float64, device=dev) if want_matrix else None
    X = torch.empty((n, N), dtype=torch.float64, device=dev) if want_X else None
    dX = torch.empty((n, N), dtype=torch.float64, device=dev) if want_dX else None
    info = torch.empty((n,), dtype=torch.int32, device=dev)
    return lam, lm, X, dX, info


def solve_gcf_batch(g, c, f, h: float, lam0=None, sigma=None, want_X=True, want_dX=True,
                    want_matrix=True, chain_len: int = 1) -> Solution:
    """K2+K3: batched ``gamma_ball_full`` from explicit ``g, c, f`` of shape ``(nsolve, N)``
    (``utils.py:1550-1624``)."""
    _lib.require_cuda()
    lib = _lib.load()
    if not (isinstance(g, torch.Tensor) and g.is_cuda):
        g = torch.as_tensor(np.asarray(g, dtype=np.float64)).cuda()
    dev = g.device
    g, c, f = _f64(g, dev, "g"), _f64(c, dev, "c"), _f64(f, dev, "f")
    if g.dim() != 2 or g.shape != c.shape or g.shape != f.shape:
        raise ValueError("g, c, f must share the shape (nsolve, N)")
    n, N = g.shape
    lam0 = None if lam0 is None else _f64(lam0, dev, "lam0")
    sigma = None if sigma is None else _f64(sigma, dev, "sigma")
    lam, lm, X, dX, info = _alloc_out(n, N, dev, want_X, want_dX, want_matrix)
    with torch.cuda.device(dev):
        rc = lib.ibs_solve_gcf_batch(_ptr(g), _ptr(c), _ptr(f), n, N, float(h), _ptr(lam0), _ptr(sigma), int(chain_len),
                                     _ptr(lam), _ptr(lm), _ptr(X), _ptr(dX), _ptr(info), _stream())
    _lib.check(rc, "ibs_solve_gcf_batch")
    return Solution(lam, lm, X, dX, info)


def solve_base_batch(base, dPdrho, theta0, h: float, nth0: Optional[int] = None, line_of_solve=None, lam0=None,
                     sigma=None, want_X=True, want_dX=True, want_matrix=True, want_gcf=False,
                     chain_len: int = 1) -> Solution:
    """K2+K3 with the coefficients formed on the fly from the eight base arrays of each field line
    (``ball_scan.py:267-268`` + ``utils.py:1560-1562``).  ``base`` is ``(nline, 8, N)`` (leading dims
    are flattened), ``theta0`` is ``(nsolve,)``; solve ``i`` uses line ``line_of_solve[i]`` or
    ``i // nth0``.  ``chain_len > 1`` warm-starts runs of consecutive solves of one line from each other
    (the batched form of the reference's start-vector chain, ``ball_scan.py:265-274``)."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = base.device
    N = base.shape[-1]
    base = _f64(base, dev, "base").reshape(-1, NBASE, N)
    dP = _f64(dPdrho, dev, "dPdrho").reshape(-1)
    theta0 = _f64(theta0, dev, "theta0").reshape(-1)
    n = theta0.numel()
    if line_of_solve is not None:
        line_of_solve = torch.as_tensor(line_of_solve).to(device=dev, dtype=torch.int32).contiguous()
        if line_of_solve.numel() != n:
            raise ValueError("line_of_solve must have one entry per solve")
    elif nth0 is None:
        if n % base.shape[0]:
            raise ValueError("give nth0 or line_of_solve")
        nth0 = n // base.shape[0]
    if line_of_solve is None and nth0 * base.shape[0] < n:
        raise ValueError("not enough field lines for the requested solves")
    lam0 = None if lam0 is None else _f64(lam0, dev, "lam0")
    sigma = None if sigma is None else _f64(sigma, dev, "sigma")
    lam, lm, X, dX, info = _alloc_out(n, N, dev, want_X, want_dX, want_matrix)
    go = [torch.empty((n, N), dtype=torch.float64, device=dev) for _ in range(3)] if want_gcf else [None] * 3
    with torch.cuda.device(dev):
        rc = lib.ibs_solve_base_batch(_ptr(base), _ptr(dP), _ptr(theta0), _ptr(line_of_solve), int(nth0 or 1), n, N,
                                      float(h), _ptr(lam0), _ptr(sigma), int(chain_len), _ptr(lam), _ptr(lm), _ptr(X),
                                      _ptr(dX), _ptr(go[0]), _ptr(go[1]), _ptr(go[2]), _ptr(info), _stream())
    _lib.check(rc, "ibs_solve_base_batch")
    return Solution(lam, lm, X, dX, info, *go)


def count_above_batch(g, c, f, h: float, lam) -> torch.Tensor:
    """Number of eigenvalues of each pencil above ``lam`` (Sturm/Newcomb node count).  ``count(0) > 0``
    is the reference's s-alpha instability test (``bishop_ball_s-alpha.py:90-115``)."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = g.device
    g, c, f = _f64(g, dev, "g"), _f64(c, dev, "c"), _f64(f, dev, "f")
    n, N = g.shape
    lam = _f64(lam, dev, "lam").reshape(-1)
    if lam.numel() == 1 and n != 1:
        lam = lam.expand(n).contiguous()
    out = torch.empty((n,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ibs_count_above_batch(_ptr(g), _ptr(c), _ptr(f), n, N, float(h), _ptr(lam), _ptr(out), _stream())
    _lib.check(rc, "ibs_count_above_batch")
    return out


# ---------------------------------------------------------------------------------------------
def adjoint_batch(lam, X, dX, f, g_p, c_p, f_p) -> torch.Tensor:
    """K4: ``d lam / d p`` for ``nparam`` perturbation triples per solve (``utils.py:1676-1680``).
    ``g_p, c_p, f_p`` are ``(nsolve, nparam, N)``; returns ``(nsolve, nparam)``."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = X.device
    n, N = X.shape
    g_p, c_p, f_p = (_f64(t, dev, "pert").reshape(n, -1, N) for t in (g_p, c_p, f_p))
    npar = g_p.shape[1]
    grad = torch.empty((n, npar), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ibs_adjoint_batch(_ptr(_f64(lam, dev, "lam")), _ptr(_f64(X, dev, "X")), _ptr(_f64(dX, dev, "dX")),
                                   _ptr(_f64(f, dev, "f")), _ptr(g_p), _ptr(c_p), _ptr(f_p), n, npar, N, _ptr(grad),
                                   _stream())
    _lib.check(rc, "ibs_adjoint_batch")
    return grad


def adjoint_sensitivities(lam, X, dX, f):
    """Per-point ``d lam/d g_j, d lam/d c_j, d lam/d f_j`` (each ``(nsolve, N)``)."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = X.device
    n, N = X.shape
    outs = [torch.empty((n, N), dtype=torch.float64, device=dev) for _ in range(3)]
    with torch.cuda.device(dev):
        rc = lib.ibs_adjoint_sensitivities(_ptr(_f64(lam, dev, "lam")), _ptr(_f64(X, dev, "X")), _ptr(_f64(dX, dev, "dX")),
                                           _ptr(_f64(f, dev, "f")), n, N, _ptr(outs[0]), _ptr(outs[1]), _ptr(outs[2]),
                                           _stream())
    _lib.check(rc, "ibs_adjoint_sensitivities")
    return tuple(outs)


def geometry_adjoint(tables: DeviceTables, alpha, theta, theta0, dPdrho, dlam_dg, dlam_dc, dlam_df, Q, phi_center: float = 0.0,
                     want_scalars: bool = False):
    """Reverse mode of K1 (``ibs_geometry_adjoint``): ``d lambda / d tab_mn (ns, 6, mnmax)`` and ``d lambda / d tab_nyq
    (ns, 7, mnmax_nyq)`` for one field line per surface, from the per-point Hellmann-Feynman sensitivities.
    ``want_scalars=True`` (``ibs_geometry_adjoint_scal``) also returns ``d lambda / d scal (ns, 8)`` (per column, the others
    held fixed; columns 5-7 are 0) and ``(d lambda / d phiedge, d lambda / d Aminor_p) (ns, 2)``."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = tables.tab_mn.device
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    f = lambda t, nm: _f64(t, dev, nm)
    alpha, theta, theta0, dP = f(alpha, "alpha").reshape(-1), f(theta, "theta").reshape(-1), f(theta0, "theta0").reshape(-1), f(dPdrho, "dPdrho").reshape(-1)
    ns, nl = tables.ns, theta.numel()
    sg, sc, sf, Q = f(dlam_dg, "dlam_dg").reshape(ns, nl), f(dlam_dc, "dlam_dc").reshape(ns, nl), f(dlam_df, "dlam_df").reshape(ns, nl), f(Q, "Q").reshape(ns)
    xm, xn, xmq, xnq = up(tables.xm), up(tables.xn), up(tables.xm_nyq), up(tables.xn_nyq)
    gmn = torch.empty_like(tables.tab_mn)
    gnq = torch.empty_like(tables.tab_nyq)
    args = (_ptr(tables.tab_mn), _ptr(tables.tab_nyq), _ptr(tables.scal), _ptr(xm), _ptr(xn), _ptr(xmq), _ptr(xnq),
            ns, xm.numel(), xmq.numel(), tables.phiedge, tables.Aminor_p, _ptr(alpha), _ptr(theta), nl,
            float(phi_center), _ptr(theta0), _ptr(dP), _ptr(sg), _ptr(sc), _ptr(sf), _ptr(Q), _ptr(gmn), _ptr(gnq))
    if want_scalars:
        gsc = torch.empty_like(tables.scal)
        ggl = torch.empty((ns, 2), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            rc = lib.ibs_geometry_adjoint_scal(*args, _ptr(gsc), _ptr(ggl), _stream())
        _lib.check(rc, "ibs_geometry_adjoint_scal")
        return gmn, gnq, gsc, ggl
    with torch.cuda.device(dev):
        rc = lib.ibs_geometry_adjoint(*args, _stream())
    _lib.check(rc, "ibs_geometry_adjoint")
    return gmn, gnq


def obj_w_grad_batch(base3, dPdrho3, theta0, h: float, del_alpha: float = 0.004, lam0=None, want_X=False):
    """Batched ``obj_w_grad`` (``utils.py:1632-1728``): ``base3`` is ``(npoint, 3, 8, N)`` holding the
    lines ``alpha - del/2, alpha, alpha + del/2``.  Returns ``(val, grad, X, dX, info)`` with
    ``val = -lam`` and ``grad = (-dlam/dalpha, -dlam/dtheta0)``."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = base3.device
    npnt, N = base3.shape[0], base3.shape[-1]
    base3 = _f64(base3, dev, "base3")
    dP3 = _f64(dPdrho3, dev, "dPdrho3").reshape(npnt, 3)
    theta0 = _f64(theta0, dev, "theta0").reshape(npnt)
    lam0 = None if lam0 is None else _f64(lam0, dev, "lam0")
    val = torch.empty((npnt,), dtype=torch.float64, device=dev)
    grad = torch.empty((npnt, 2), dtype=torch.float64, device=dev)
    X = torch.empty((npnt, N), dtype=torch.float64, device=dev) if want_X else None
    dX = torch.empty((npnt, N), dtype=torch.float64, device=dev) if want_X else None
    info = torch.empty((npnt,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ibs_obj_w_grad_batch(_ptr(base3), _ptr(dP3), _ptr(theta0), npnt, N, float(h), float(del_alpha),
                                      _ptr(lam0), _ptr(val), _ptr(grad), _ptr(X), _ptr(dX), _ptr(info), _stream())
    _lib.check(rc, "ibs_obj_w_grad_batch")
    return val, grad, X, dX, info


def obj_w_grad_tangent_batch(base, dbase, dPdrho, ddPdrho, theta0, h: float, lam0=None, want_X=False):
    """``obj_w_grad`` with the exact alpha-derivative (``ibs_obj_w_grad_tangent_batch``): ``base`` and ``dbase`` are
    ``(npoint, 8, N)`` (one line per point and its alpha-tangent, from ``geometry_tangent_batch``), ``dPdrho`` and
    ``ddPdrho`` ``(npoint,)``.  Returns ``(val, grad, X, dX, info)`` as ``obj_w_grad_batch``; ``val``, ``grad[:, 1]``, ``X``
    and ``info`` are its bits on the same centre lines, ``grad[:, 0]`` is the chain rule instead of a central difference."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = base.device
    N = base.shape[-1]
    base = _f64(base, dev, "base").reshape(-1, NBASE, N)
    npnt = base.shape[0]
    dbase = _f64(dbase, dev, "dbase").reshape(npnt, NBASE, N)
    dP = _f64(dPdrho, dev, "dPdrho").reshape(npnt)
    ddP = _f64(ddPdrho, dev, "ddPdrho").reshape(npnt)
    theta0 = _f64(theta0, dev, "theta0").reshape(npnt)
    lam0 = None if lam0 is None else _f64(lam0, dev, "lam0")
    val = torch.empty((npnt,), dtype=torch.float64, device=dev)
    grad = torch.empty((npnt, 2), dtype=torch.float64, device=dev)
    X = torch.empty((npnt, N), dtype=torch.float64, device=dev) if want_X else None
    dX = torch.empty((npnt, N), dtype=torch.float64, device=dev) if want_X else None
    info = torch.empty((npnt,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ibs_obj_w_grad_tangent_batch(_ptr(base), _ptr(dbase), _ptr(dP), _ptr(ddP), _ptr(theta0), npnt, N, float(h),
                                              _ptr(lam0), _ptr(val), _ptr(grad), _ptr(X), _ptr(dX), _ptr(info), _stream())
    _lib.check(rc, "ibs_obj_w_grad_tangent_batch")
    return val, grad, X, dX, info


class RefineState:
    """Device-resident state of the batched refinement (``ibs_refine_init`` / ``ibs_refine_step``): ``n`` independent
    2-D box-constrained problems advanced in lock step.  ``alphas3 (n, 3)`` and ``theta0 (n,)`` always hold the NEXT trial
    points in the layout ``geometry_batch`` / ``obj_w_grad_batch`` take."""

    def __init__(self, alpha0, theta0, bounds=((0.0, float(np.pi)), (0.0, 0.5 * float(np.pi))), del_alpha: float = 0.004):
        _lib.require_cuda()
        lib = _lib.load()
        dev = alpha0.device
        self.n = alpha0.numel()
        self.del_alpha = float(del_alpha)
        self.nstate = lib.ibs_refine_state_doubles()
        self.state = torch.zeros((self.n, self.nstate), dtype=torch.float64, device=dev)
        self.alphas3 = torch.empty((self.n, 3), dtype=torch.float64, device=dev)
        self.theta0 = torch.empty((self.n,), dtype=torch.float64, device=dev)
        self.nactive = torch.zeros((1,), dtype=torch.int32, device=dev)
        a0, t0 = _f64(alpha0, dev, "alpha0").reshape(-1), _f64(theta0, dev, "theta0").reshape(-1)
        with torch.cuda.device(dev):
            rc = lib.ibs_refine_init(_ptr(self.state), self.n, _ptr(a0), _ptr(t0), float(bounds[0][0]), float(bounds[0][1]),
                                     float(bounds[1][0]), float(bounds[1][1]), self.del_alpha, _ptr(self.alphas3), _ptr(self.theta0),
                                     _stream())
        _lib.check(rc, "ibs_refine_init")

    def step(self, val, grad, info, ftol: float, gtol: float, maxiter: int):
        lib = _lib.load()
        with torch.cuda.device(self.state.device):
            rc = lib.ibs_refine_step(_ptr(self.state), self.n, _ptr(val), _ptr(grad), _ptr(info), float(ftol), float(gtol), int(maxiter),
                                     self.del_alpha, _ptr(self.alphas3), _ptr(self.theta0), _ptr(self.nactive), _stream())
        _lib.check(rc, "ibs_refine_step")

    # views into the state (see include/ibs_b200.h)
    x = property(lambda self: self.state[:, 0:2])
    fun = property(lambda self: self.state[:, 2])
    status = property(lambda self: self.state[:, 18])
    why = property(lambda self: self.state[:, 19])
    nit = property(lambda self: self.state[:, 20])
    nfev = property(lambda self: self.state[:, 21])


def scan_argmax(gamma):
    """Per-surface arg-max over the flattened ``(alpha, theta0)`` grid with the reference's guards
    (``ball_scan.py:279-295``).  ``gamma`` is ``(ns, ...)``; returns ``(val, flat_idx, sigma0)``;
    ``flat_idx = -1`` encodes the all-zero guard."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = gamma.device
    ns = gamma.shape[0]
    gm = _f64(gamma, dev, "gamma").reshape(ns, -1)
    val = torch.empty((ns,), dtype=torch.float64, device=dev)
    idx = torch.empty((ns,), dtype=torch.int32, device=dev)
    sig = torch.empty((ns,), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ibs_scan_argmax(_ptr(gm), ns, gm.shape[1], _ptr(val), _ptr(idx), _ptr(sig), _stream())
    _lib.check(rc, "ibs_scan_argmax")
    return val, idx, sig


def scan_solve_argmax(base, dPdrho, theta0, h: float, nth0: int, lines_per_surface: int, sigma=None, want_X=False,
                      want_dX=False, chain_len: int = 1, best_out: Optional[torch.Tensor] = None):
    """The coarse scan of ``ball_scan.py:248-295`` in one call: K2+K3 for ``nline x nth0`` solves (theta0 fastest) with
    the guarded per-surface arg-max fused into the solver kernel.  Returns ``(Solution, best, sigma0)``;
    ``best`` is ``(nsurf, 2)`` = packed ``(max, flat index as a double; -1 = all-zero guard)`` -- pass a slice of a
    preallocated gather buffer as ``best_out`` and it IS the send slot of the all-gather."""
    _lib.require_cuda()
    lib = _lib.load()
    dev = base.device
    N = base.shape[-1]
    base = _f64(base, dev, "base").reshape(-1, NBASE, N)
    nline = base.shape[0]
    dP = _f64(dPdrho, dev, "dPdrho").reshape(-1)
    theta0 = _f64(theta0, dev, "theta0").reshape(-1)
    n = nline * int(nth0)
    if theta0.numel() != n or nline % int(lines_per_surface):
        raise ValueError("theta0 must hold nline * nth0 values and nline must be a multiple of lines_per_surface")
    nsurf = nline // int(lines_per_surface)
    sigma = None if sigma is None else _f64(sigma, dev, "sigma")
    lam, _, X, dX, info = _alloc_out(n, N, dev, want_X, want_dX, False)
    if best_out is None:
        best_out = torch.empty((nsurf, 2), dtype=torch.float64, device=dev)
    elif best_out.dtype != torch.float64 or best_out.numel() != 2 * nsurf or not best_out.is_contiguous():
        raise ValueError("best_out must be a contiguous float64 tensor of shape (nsurf, 2)")
    sig0 = torch.empty((nsurf,), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        rc = lib.ibs_scan_solve_argmax(_ptr(base), _ptr(dP), _ptr(theta0), int(nth0), nline, int(lines_per_surface), N,
                                       float(h), _ptr(sigma), int(chain_len), _ptr(lam), _ptr(X), _ptr(dX), _ptr(info),
                                       _ptr(best_out), _ptr(sig0), _stream())
    _lib.check(rc, "ibs_scan_solve_argmax")
    return Solution(lam, None, X, dX, info), best_out, sig0


def scan_host(st: SurfaceTables, alpha, theta0, theta, want_xbest: bool = False, out=None, want_xall: bool = False):
    """End-to-end coarse scan with HOST (numpy) buffers through ``ibs_scan_host``: H2D of the tables,
    K1 + K3 (fused arg-max), D2H of the results.  Returns ``(gamma (ns, nalpha, nth0), val, idx, sigma0, nbad)``
    (+ ``xbest (ns, nl)``, the eigenfunction at each surface's maximum, when ``want_xbest``; + ``xall
    (ns, nalpha, nth0, nl)``, the eigenfunction of EVERY solve, when ``want_xall``).  ``out`` may carry
    preallocated (e.g. pinned) result arrays ``dict(gamma=, val=, idx=, sigma0=, xbest=, xall=)``."""
    _lib.require_cuda()
    lib = _lib.load()
    c = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    tab_mn, tab_nyq, scal = c(st.tab_mn), c(st.tab_nyq), c(st.scal)
    xm, xn, xmq, xnq = c(st.xm), c(st.xn), c(st.xm_nyq), c(st.xn_nyq)
    alpha, theta0, theta = c(alpha), c(theta0), c(theta)
    ns, na, nt, nl = tab_mn.shape[0], alpha.size, theta0.size, theta.size
    out = out or {}
    gamma = out.get("gamma") if out.get("gamma") is not None else np.empty((ns, na, nt))
    val = out.get("val") if out.get("val") is not None else np.empty(ns)
    sig = out.get("sigma0") if out.get("sigma0") is not None else np.empty(ns)
    idx = out.get("idx") if out.get("idx") is not None else np.empty(ns, dtype=np.int32)
    xbest = xall = None
    if want_xbest:
        xbest = out.get("xbest") if out.get("xbest") is not None else np.empty((ns, nl))
    if want_xall:
        xall = out.get("xall") if out.get("xall") is not None else np.empty((ns, na, nt, nl))
    import ctypes
    nbad = ctypes.c_int(0)
    p = lambda a: a.ctypes.data
    rc = lib.ibs_scan_host(p(tab_mn), p(tab_nyq), p(scal), p(xm), p(xn), p(xmq), p(xnq), ns, len(xm), len(xmq),
                           float(st.phiedge), float(st.Aminor_p), p(alpha), na, p(theta0), nt, p(theta), nl,
                           grid_spacing(theta), p(gamma), p(val), p(idx), p(sig),
                           None if xbest is None else p(xbest), None if xall is None else p(xall), ctypes.addressof(nbad))
    _lib.check(rc, "ibs_scan_host")
    res = (gamma, val, idx, sig, nbad.value)
    if want_xbest:
        res = res + (xbest,)
    if want_xall:
        res = res + (xall,)
    return res
