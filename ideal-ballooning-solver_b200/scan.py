"""Growth-rate scan over (surface s, field-line label alpha, ballooning angle theta0).

Batched re-expression of the loops of ``/root/reference/ball_scan.py:196-339``: the reference runs
one MPI group per surface and one rank per alpha stripe (``ball_scan.py:172-194,248-252``) and
gathers three doubles per surface at the end (``:341-347``).  Here every (s, alpha) field line and
every (s, alpha, theta0) solve is one element of a batched launch; surfaces are sharded in
contiguous blocks over ranks (one process per GPU) and the only exchange is one all-gather of the
per-surface maxima.
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import numpy as np
import torch

from . import engine
from .tables import SurfaceTables

# reference defaults (ball_scan.py:197,201,223-226; utils.py:1639; ball_scan.py:313)
THETA_FAC = 4
NTHETA0_GUESS = 15
NALPHA_GUESS = 24
DEL_ALPHA = 0.004


def scan_theta_grid(mpol: int, ntor: int, theta_fac: int = THETA_FAC) -> np.ndarray:
    """The theta grid of ``ball_scan.py:201-208`` (``ntheta`` odd)."""
    ntheta = int(2 * mpol * theta_fac) + 1 if ntor == 0 else int(2 * mpol * ntor * theta_fac) + 1
    return np.linspace(-theta_fac * np.pi, theta_fac * np.pi, ntheta)


def chain_length(nth0: int, cap: int = 16) -> int:
    """Warm-start run length over consecutive theta0 of one field line (``ball_scan.py:265-274`` chains its
    start vector through the same loop): the largest divisor of ``nth0`` not above ``cap``."""
    k = min(int(nth0), cap)
    while k > 1 and nth0 % k:
        k -= 1
    return max(k, 1)


def shard_range(n: int, rank: int, world: int):
    """Contiguous block of ``range(n)`` owned by ``rank`` (sizes differ by at most one)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


@dataclasses.dataclass
class ScanResult:
    gamma: torch.Tensor            # (ns_local, nalpha, nth0)
    val: torch.Tensor              # (ns_local,)   max over the grid (ball_scan.py:279-295)
    idx: torch.Tensor              # (ns_local,)   flat (alpha, theta0) index of the maximum, -1 = all-zero guard
    sigma0: torch.Tensor           # (ns_local,)   1.3 |max| + 0.05
    alpha_guess: torch.Tensor      # (ns_local,)
    theta0_guess: torch.Tensor     # (ns_local,)
    X: Optional[torch.Tensor]      # (ns_local, nalpha, nth0, nl) eigenfunctions (if requested)
    info: torch.Tensor
    geometry: engine.Geometry


def coarse_scan(tables: engine.DeviceTables, alpha, theta0, theta, want_X: bool = False,
                lam0=None, best_out: Optional[torch.Tensor] = None) -> ScanResult:
    """Coarse (alpha, theta0) grid of every surface in ``tables`` (``ball_scan.py:248-295``): K1 for
    ``ns x nalpha`` field lines, K2+K3 for ``ns x nalpha x nth0`` solves, guarded arg-max."""
    dev = tables.tab_mn.device
    alpha_t = torch.as_tensor(np.asarray(alpha, dtype=np.float64)).to(dev) if not isinstance(alpha, torch.Tensor) else alpha
    theta0_t = torch.as_tensor(np.asarray(theta0, dtype=np.float64)).to(dev) if not isinstance(theta0, torch.Tensor) else theta0
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    geo = engine.geometry_batch(tables, alpha_t, theta_np)
    ns, na, nt = tables.ns, alpha_t.shape[-1], theta0_t.numel()
    th0 = theta0_t.repeat(ns * na)
    if lam0 is None:
        sol, best, sig = engine.scan_solve_argmax(geo.base, geo.dPdrho, th0, engine.grid_spacing(theta_np), nt, na, want_X=want_X,
                                                  chain_len=chain_length(nt), best_out=best_out)
        gamma = sol.lam.reshape(ns, na, nt)
        val, idx = best[:, 0], best[:, 1].to(torch.int32)
    else:
        sol = engine.solve_base_batch(geo.base, geo.dPdrho, th0, engine.grid_spacing(theta_np), nth0=nt, lam0=lam0,
                                      want_X=want_X, want_dX=False, want_matrix=False, chain_len=chain_length(nt))
        gamma = sol.lam.reshape(ns, na, nt)
        val, idx, sig = engine.scan_argmax(gamma)
        if best_out is not None:
            best_out[:, 0] = val
            best_out[:, 1] = idx.to(torch.float64)
    safe = idx.clamp(min=0).long()
    ia, it = safe // nt, safe % nt
    if alpha_t.dim() == 2:
        a_guess = alpha_t.gather(1, ia[:, None])[:, 0]
    else:
        a_guess = alpha_t[ia]
    t_guess = theta0_t[it]
    zero = idx < 0          # ball_scan.py:279-282: alpha_guess = theta0_guess = 0
    a_guess = torch.where(zero, torch.zeros_like(a_guess), a_guess)
    t_guess = torch.where(zero, torch.zeros_like(t_guess), t_guess)
    X = sol.X.reshape(ns, na, nt, -1) if want_X else None
    return ScanResult(gamma, val, idx, sig, a_guess, t_guess, X, sol.info, geo)


@dataclasses.dataclass
class MarginalScanResult:
    kappa: torch.Tensor            # (ns, nalpha, nth0) critical pressure-gradient factor kappa* of every solve
    kappa_min: torch.Tensor        # (ns,) smallest kappa* of each surface (< 1: unstable as given)
    idx: torch.Tensor              # (ns,) its flat (alpha, theta0) index (first minimum)
    alpha_crit: torch.Tensor       # (ns,)
    theta0_crit: torch.Tensor      # (ns,)
    X: Optional[torch.Tensor]      # (ns, nl) null vector of each surface's minimum (if requested)
    info: torch.Tensor             # (ns, nalpha, nth0) sweeps | flags << 16
    geometry: engine.Geometry


def marginal_scan(tables: engine.DeviceTables, alpha, theta0, theta, kappa_max: float = 1e3, rtol: float = 1e-12,
                  want_X: bool = False) -> MarginalScanResult:
    """Distance of every surface from ballooning instability on the coarse (alpha, theta0) grid: K1 for ``ns x nalpha``
    field lines, ``engine.marginal_batch`` for every solve, and per surface the smallest kappa* with its (alpha, theta0).
    The reduction is ``engine.scan_argmax(-kappa)``: first index among equal values, and kappa* > 0 keeps its all-zero
    guard from firing.  +inf (stable up to ``kappa_max``) enters as the largest double, so a surface stable everywhere
    reports ``kappa_min = inf`` at index 0; a NaN (bad input) gives ``kappa_min = nan`` and index -2."""
    dev = tables.tab_mn.device
    alpha_t = torch.as_tensor(np.asarray(alpha, dtype=np.float64)).to(dev) if not isinstance(alpha, torch.Tensor) else alpha
    theta0_t = torch.as_tensor(np.asarray(theta0, dtype=np.float64)).to(dev) if not isinstance(theta0, torch.Tensor) else theta0
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    geo = engine.geometry_batch(tables, alpha_t, theta_np)
    ns, na, nt = tables.ns, alpha_t.shape[-1], theta0_t.numel()
    h = engine.grid_spacing(theta_np)
    m = engine.marginal_batch(geo.base, geo.dPdrho, theta0_t.repeat(ns * na), h, nth0=nt, kappa_max=kappa_max, rtol=rtol)
    kappa = m.kappa.reshape(ns, na, nt)
    big = torch.finfo(torch.float64).max
    neg, idx, _ = engine.scan_argmax((-kappa).clamp(min=-big))
    kmin = torch.where(neg == -big, torch.full_like(neg, float("inf")), -neg)
    safe = idx.clamp(min=0).long()
    ia, it = safe // nt, safe % nt
    a_crit = alpha_t.gather(1, ia[:, None])[:, 0] if alpha_t.dim() == 2 else alpha_t[ia]
    X = None
    if want_X:
        line = torch.arange(ns, device=dev, dtype=torch.int64) * na + ia
        X = engine.marginal_batch(geo.base, geo.dPdrho, theta0_t[it], h, line_of_solve=line, kappa_max=kappa_max, rtol=rtol,
                                  want_X=True).X
    return MarginalScanResult(kappa, kmin, idx, a_crit, theta0_t[it], X, m.info.reshape(ns, na, nt), geo)


class SurfaceGather:
    """The one exchange step of the scan (replaces the three ``MPI.Gather`` of ``ball_scan.py:345-347``) with NO kernel
    but the collective itself: the solver writes each local surface's packed ``(max, index)`` pair straight into this
    object's send slot (``engine.scan_solve_argmax(..., best_out=g.send)``), and ``g.exchange()`` is one
    ``all_gather_into_tensor`` into a preallocated ``(world, nmax, 2)`` buffer.  Works with NCCL (GPU tensors) and gloo
    (CPU tensors).  Ranks own contiguous blocks of surfaces (``shard_range``); shorter blocks leave their tail rows unused."""

    def __init__(self, ns_total: int, device, group=None):
        import torch.distributed as dist
        self.group = group
        self.dist = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.world = dist.get_world_size(group) if self.dist else 1
        self.rank = dist.get_rank(group) if self.dist else 0
        self.sizes = [shard_range(ns_total, r, self.world) for r in range(self.world)]
        self.nmax = max(1, max(hi - lo for lo, hi in self.sizes))
        lo, hi = self.sizes[self.rank]
        self.nlocal = hi - lo
        self.recv = torch.zeros((self.world, self.nmax, 2), dtype=torch.float64, device=device)
        self._send_full = self.recv[self.rank] if not self.dist else torch.zeros((self.nmax, 2), dtype=torch.float64, device=device)
        self.send = self._send_full[: self.nlocal]          # (nlocal, 2) contiguous view: the solver's best_out

    def exchange(self, async_op: bool = False) -> torch.Tensor:
        """All-gather the send slots; returns the ``(world, nmax, 2)`` buffer (no copy, no cast).  ``async_op=True``: the
        collective is only enqueued (it starts when the work already queued on the current stream -- the solver that fills the
        send slot -- is done) and the current stream does NOT wait for it: the next scan's kernels overlap it.  Call ``wait()``
        before reading ``recv`` or refilling ``send`` (use two ``SurfaceGather`` objects alternately to keep scanning)."""
        if self.dist:
            import torch.distributed as dist
            self.wait()
            w = dist.all_gather_into_tensor(self.recv.view(-1), self._send_full.view(-1), group=self.group, async_op=async_op)
            self._work = w if async_op else None
        return self.recv

    def wait(self):
        """Make the current stream wait for the pending asynchronous exchange (no-op when there is none)."""
        w = getattr(self, "_work", None)
        if w is not None:
            w.wait()
            self._work = None

    def unpack(self):
        """``(val (ns_total,), idx (ns_total,) int32)`` in surface order (host-side convenience, not on the timed path)."""
        vals = torch.cat([self.recv[r, : hi - lo, 0] for r, (lo, hi) in enumerate(self.sizes)])
        idxs = torch.cat([self.recv[r, : hi - lo, 1] for r, (lo, hi) in enumerate(self.sizes)]).to(torch.int32)
        return vals, idxs


def gather_surface_maxima(val: torch.Tensor, idx: torch.Tensor, ns_total: int, group=None):
    """All-gather per-surface ``(val, idx)`` pairs of every rank's contiguous block of surfaces (convenience form on
    separate arrays; the scan itself uses ``SurfaceGather``, whose send slot the solver kernel fills directly)."""
    g = SurfaceGather(ns_total, val.device, group)
    if g.world == 1:
        return val, idx
    g.send[:, 0] = val
    g.send[:, 1] = idx.to(torch.float64)
    g.exchange()
    return g.unpack()


def sharded_coarse_scan(st: SurfaceTables, alpha, theta0, theta, device=None, want_X=False, group=None):
    """Shard the surfaces of ``st`` over the ranks of ``group`` (or run everything when not
    distributed), scan the local block and all-gather the per-surface maxima.  Returns
    ``(local ScanResult, (lo, hi), val_all, idx_all)``."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    else:
        rank, world = 0, 1
    lo, hi = shard_range(st.ns, rank, world)
    device = device or torch.device("cuda", torch.cuda.current_device())
    gather = SurfaceGather(st.ns, device, group)
    res = None
    if hi > lo:
        dt = engine.DeviceTables.from_host(st.select(np.arange(lo, hi)), device)
        res = coarse_scan(dt, alpha, theta0, theta, want_X=want_X, best_out=gather.send)
    # (more ranks than surfaces: a rank with nothing to scan still takes part in the exchange)
    gather.exchange()
    val_all, idx_all = gather.unpack()
    return res, (lo, hi), val_all, idx_all


# ---------------------------------------------------------------------------------------------
# Refinement of the coarse maxima and the drop-in driver (SURVEY.md section 8 row f2)
# ---------------------------------------------------------------------------------------------
class _BatchedObjective:
    """Lets ``ns`` independent ``scipy.optimize.minimize`` instances (one Python thread per surface, exactly the
    reference's optimiser and options, ``ball_scan.py:305-314``) share ONE batched GPU evaluation of
    ``obj_w_grad`` per round: every thread posts its ``(alpha, theta0)`` and blocks; the thread that completes
    the round runs K1 (three field lines per point) + K3 + K4 for all pending points and wakes the others."""

    def __init__(self, tables: engine.DeviceTables, theta_np, del_alpha=DEL_ALPHA):
        import threading
        self.tables, self.theta = tables, theta_np
        self.h = engine.grid_spacing(theta_np)
        self.del_alpha = del_alpha
        self.cv = threading.Condition()
        self.active = set()
        self.pending = {}
        self.results = {}
        self.nbatches = 0
        self.nevals = 0

    def start(self, ids):
        self.active = set(ids)

    def _run_batch(self):
        ids = sorted(self.pending)
        xs = np.array([self.pending[i] for i in ids], dtype=np.float64)
        dev = self.tables.tab_mn.device
        sel = torch.as_tensor(ids, device=dev, dtype=torch.long)
        sub = dataclasses.replace(self.tables, tab_mn=self.tables.tab_mn.index_select(0, sel).contiguous(),
                                  tab_nyq=self.tables.tab_nyq.index_select(0, sel).contiguous(),
                                  scal=self.tables.scal.index_select(0, sel).contiguous())
        d = self.del_alpha
        alphas = np.stack([xs[:, 0] - 0.5 * d, xs[:, 0], xs[:, 0] + 0.5 * d], axis=1)        # utils.py:1641-1646
        geo = engine.geometry_batch(sub, torch.from_numpy(alphas).to(dev), self.theta)
        val, grad, _, _, info = engine.obj_w_grad_batch(geo.base, geo.dPdrho, torch.from_numpy(xs[:, 1].copy()).to(dev),
                                                        self.h, del_alpha=d)
        val, grad, info = val.cpu().numpy(), grad.cpu().numpy(), info.cpu().numpy()
        for k, i in enumerate(ids):
            self.results[i] = (float(val[k]), grad[k].copy(), int(info[k]) >> 16)
        self.pending.clear()
        self.nbatches += 1
        self.nevals += len(ids)

    def _run_batch_guarded(self):
        """Run the pending round; a failure (CUDA error, bad input, ...) becomes the result of EVERY pending surface, so
        that no waiting thread is left behind (each of them re-raises it)."""
        try:
            self._run_batch()
        except BaseException as e:          # noqa: BLE001 - handed to the waiting threads
            for i in list(self.pending):
                self.results[i] = e
            self.pending.clear()
        self.cv.notify_all()

    def evaluate(self, i, x):
        with self.cv:
            self.pending[i] = (float(x[0]), float(x[1]))
            if len(self.pending) == len(self.active):
                self._run_batch_guarded()
            else:
                while i not in self.results:
                    self.cv.wait()
            res = self.results.pop(i)
        if isinstance(res, BaseException):
            raise RuntimeError("obj_w_grad: batched evaluation failed (surface %d)" % i) from res
        val, grad, flags = res
        if flags & (engine.FLAG_NOT_CONVERGED | engine.FLAG_BAD_INPUT):
            raise RuntimeError("obj_w_grad: eigen-solve failed on surface %d" % i)
        return val, grad

    def finish(self, i):
        with self.cv:
            self.active.discard(i)
            self.pending.pop(i, None)
            if self.pending and len(self.pending) == len(self.active):
                self._run_batch_guarded()


@dataclasses.dataclass
class RefineResult:
    alpha: np.ndarray          # (ns,) alpha at the refined maximum
    theta0: np.ndarray         # (ns,)
    fun: np.ndarray            # (ns,) -lambda at the optimiser's last point
    nit: np.ndarray
    nfev: np.ndarray
    success: np.ndarray
    nbatches: int              # batched GPU evaluations issued (vs sum(nfev) one-at-a-time in the reference)


def refine_maxima(tables: engine.DeviceTables, alpha_guess, theta0_guess, theta, maxiter: int = 30, ftol: float = 5.0e-11,
                  gtol: float = 2.0e-08, method: str = "device", max_rounds: int = 200, sync_every: int = 4,
                  alpha_derivative: str = "fd") -> RefineResult:
    """Refinement of every surface's coarse maximum (``ball_scan.py:305-314``: ``scipy.optimize.minimize(obj_w_grad,
    x0=(alpha_guess, theta0_guess), jac=True, bounds=((0, pi), (0, pi/2)), options={ftol, gtol, maxiter})``).

    ``method="device"`` (default): the batched projected quasi-Newton method of ``csrc/ibs_refine_core.cuh`` -- all surfaces in
    lock step, the optimiser state resident on the GPU; one round = K1 (three field lines per surface) + K2/K3 + K4
    (``ibs_obj_w_grad_batch``) + ``ibs_refine_step``, no host arithmetic; the host only polls the count of running problems
    every ``sync_every`` rounds.  ``method="scipy"``: the reference's own optimiser, one Python thread per surface around the
    same batched evaluations (kept as the cross-check).

    ``alpha_derivative`` (device method): ``"fd"`` (default) is the reference's central difference of (g, c, f) over the
    lines ``alpha -+ 0.002`` (``utils.py:1707-1725``, three field lines per surface and round); ``"exact"`` takes K1 and its
    alpha-tangent on the centre line only (``engine.geometry_tangent_batch`` + ``engine.obj_w_grad_tangent_batch``): the exact
    derivative, one field line per surface and round."""
    if alpha_derivative not in ("fd", "exact"):
        raise ValueError("alpha_derivative must be 'fd' or 'exact'")
    if method == "scipy" and alpha_derivative != "fd":
        raise ValueError("method='scipy' evaluates the reference's obj_w_grad: alpha_derivative must be 'fd'")
    if method == "scipy":
        return _refine_maxima_scipy(tables, alpha_guess, theta0_guess, theta, maxiter, ftol, gtol)
    if method != "device":
        raise ValueError("method must be 'device' or 'scipy'")
    dev = tables.tab_mn.device
    ns = tables.ns
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    theta_d = torch.from_numpy(theta_np).to(dev)
    h = engine.grid_spacing(theta_np)
    as_dev = lambda a: (a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a, dtype=np.float64))).to(dev).reshape(ns)
    st = engine.RefineState(as_dev(alpha_guess), as_dev(theta0_guess), del_alpha=DEL_ALPHA)
    rounds = 0
    while rounds < max_rounds:
        for _ in range(sync_every):
            if alpha_derivative == "exact":
                geo = engine.geometry_tangent_batch(tables, st.alphas3[:, 1:2], theta_d)     # the centre line alpha
                val, grad, _, _, info = engine.obj_w_grad_tangent_batch(geo.base, geo.dbase, geo.dPdrho, geo.ddPdrho, st.theta0, h)
            else:
                geo = engine.geometry_batch(tables, st.alphas3, theta_d)                      # utils.py:1641-1646: alpha -+ del/2
                val, grad, _, _, info = engine.obj_w_grad_batch(geo.base, geo.dPdrho, st.theta0, h, del_alpha=DEL_ALPHA)
            st.step(val, grad, info, ftol, gtol, maxiter)
            rounds += 1
        if int(st.nactive.item()) == 0:
            break
    S = st.state.cpu().numpy()
    why = S[:, 19].astype(int)
    if np.any(why == 5):
        raise RuntimeError("obj_w_grad: eigen-solve failed at the starting point of surface(s) %s" % np.flatnonzero(why == 5).tolist())
    return RefineResult(alpha=S[:, 0].copy(), theta0=S[:, 1].copy(), fun=S[:, 2].copy(), nit=S[:, 20].astype(int),
                        nfev=S[:, 21].astype(int), success=np.isin(why, (1, 2, 3, 4)), nbatches=rounds)


def _refine_maxima_scipy(tables: engine.DeviceTables, alpha_guess, theta0_guess, theta, maxiter: int = 30, ftol: float = 5.0e-11,
                         gtol: float = 2.0e-08) -> RefineResult:
    """The reference's optimiser itself (scipy L-BFGS-B with its options), one Python thread per surface, the objective
    evaluated on the GPU for all surfaces at once (cross-check of the device method)."""
    import threading
    from scipy.optimize import minimize
    ns = tables.ns
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    a0 = np.asarray(alpha_guess.cpu() if isinstance(alpha_guess, torch.Tensor) else alpha_guess, dtype=np.float64).reshape(ns)
    t0 = np.asarray(theta0_guess.cpu() if isinstance(theta0_guess, torch.Tensor) else theta0_guess, dtype=np.float64).reshape(ns)
    obj = _BatchedObjective(tables, theta_np)
    obj.start(range(ns))
    out = [None] * ns
    err = [None] * ns

    def worker(i):
        try:
            out[i] = minimize(lambda x: obj.evaluate(i, x), x0=(a0[i], t0[i]), jac=True,
                              bounds=((0.0, np.pi), (0.0, 0.5 * np.pi)),
                              options={"ftol": ftol, "gtol": gtol, "maxiter": maxiter})
        except Exception as e:          # keep the other surfaces going
            err[i] = e
        finally:
            obj.finish(i)

    threads = [threading.Thread(target=worker, args=(i,), daemon=True) for i in range(ns)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in err:
        if e is not None:
            raise e
    return RefineResult(alpha=np.array([o.x[0] for o in out]), theta0=np.array([o.x[1] for o in out]),
                        fun=np.array([float(o.fun) for o in out]), nit=np.array([o.nit for o in out]),
                        nfev=np.array([o.nfev for o in out]), success=np.array([bool(o.success) for o in out]),
                        nbatches=obj.nbatches)


@dataclasses.dataclass
class BallScanResult:
    gamma: np.ndarray          # (ns,) maximum growth rate per surface        (ball_gam<dof>.npy row)
    theta0: np.ndarray         # (ns,)                                         (ball_theta0<dof>.npy row)
    alpha: np.ndarray          # (ns,)                                         (ball_alpha<dof>.npy row)
    gamma_coarse: np.ndarray   # (ns, nalpha, ntheta0) coarse grid
    X: np.ndarray              # (ns, nl) eigenfunction at the optimum
    refine: Optional[RefineResult]


def ball_scan(st: SurfaceTables, theta=None, mpol: Optional[int] = None, ntor: Optional[int] = None,
              nalpha_guess: int = NALPHA_GUESS, ntheta0_guess: int = NTHETA0_GUESS, refine: bool = True,
              device=None, refine_method: str = "device", alpha_derivative: str = "fd") -> BallScanResult:
    """The numerical section of ``ball_scan.py:196-339`` for all surfaces of ``st`` at once:
    coarse 24 x 15 (alpha, theta0) grid (``:223-274``) -> guarded arg-max (``:279-295``) -> L-BFGS-B refinement
    from the coarse maximum with the adjoint gradient (``:305-314``) -> eigenpair at the optimum (``:322-339``).
    ``alpha_derivative`` is passed to ``refine_maxima``."""
    if theta is None:
        theta = scan_theta_grid(mpol, ntor)
    theta = np.asarray(theta, dtype=np.float64)
    device = device or torch.device("cuda", torch.cuda.current_device())
    dt = engine.DeviceTables.from_host(st, device)
    alpha_scan = np.linspace(0, np.pi, nalpha_guess)                      # ball_scan.py:225-226
    theta0_scan = np.linspace(0.0, 0.5 * np.pi, ntheta0_guess)
    res = coarse_scan(dt, alpha_scan, theta0_scan, theta)
    a_star, t_star = res.alpha_guess.cpu().numpy(), res.theta0_guess.cpu().numpy()
    ref = None
    if refine:
        ref = refine_maxima(dt, a_star, t_star, theta, method=refine_method, alpha_derivative=alpha_derivative)
        a_star, t_star = ref.alpha, ref.theta0
    # ball_scan.py:322-339: geometry and eigenpair at the optimum
    geo = engine.geometry_batch(dt, torch.from_numpy(a_star[:, None].copy()).to(device), theta)
    sol = engine.solve_base_batch(geo.base, geo.dPdrho, torch.from_numpy(t_star.copy()).to(device), engine.grid_spacing(theta),
                                  nth0=1, want_dX=False, want_matrix=False)
    return BallScanResult(gamma=sol.lam.cpu().numpy(), theta0=t_star, alpha=a_star, gamma_coarse=res.gamma.cpu().numpy(),
                          X=sol.X.cpu().numpy(), refine=ref)


def _gcf_exact(geo, theta0: torch.Tensor):
    """``g, c, f`` (``utils.py:1560-1562``) of one solve per field line of ``geo`` at ``theta0`` (``ball_scan.py:267-268``),
    as torch expressions in the reference's operation order.  ``geo.base`` is ``(nline, 8, N)`` flattened."""
    b = geo.base.reshape(-1, engine.NBASE, geo.base.shape[-1])
    B, gp = b[:, engine.BASE_NAMES.index("bmag")], b[:, engine.BASE_NAMES.index("gradpar_theta_pest")].abs()
    t0 = theta0.reshape(-1, 1)
    cv = b[:, engine.BASE_NAMES.index("cvdrift")] + t0 * b[:, engine.BASE_NAMES.index("cvdrift0")]
    gd = (b[:, engine.BASE_NAMES.index("gds2")] + 2 * t0 * b[:, engine.BASE_NAMES.index("gds21")]
          + t0 ** 2 * b[:, engine.BASE_NAMES.index("gds22")])
    dP = geo.dPdrho.reshape(-1, 1)
    return gp * gd / B, -1 * dP * cv * 1 / (gp * B), gd / B ** 2 * 1 / (gp * B)


@dataclasses.dataclass
class GammaSensitivity:
    gamma: np.ndarray          # (ns,) growth rate of the base equilibrium at (alpha*, theta0*)
    dgamma: np.ndarray         # (ndof, ns) first-order change for every perturbed equilibrium
    X: np.ndarray              # (ns, nl) eigenfunction of the base equilibrium


def hellmann_feynman_gamma(tables0: engine.DeviceTables, tables_pert, alpha_star, theta0_star, theta) -> GammaSensitivity:
    """SURVEY.md section 8 row f3 (second half): the change of every surface's maximum growth rate under perturbed
    equilibria WITHOUT re-scanning them.  The reference re-runs the whole scan for each of the ``ndofs + 1`` equilibria
    of a finite-difference Jacobian (``sims_runner_NCSX.py:245-262``); to first order the change of the maximum is the
    change at fixed ``(alpha*, theta0*)`` (the maximum is stationary in both) and, at fixed eigenfunction, the
    Hellmann-Feynman contraction the reference itself uses for its (alpha, theta0) gradients (``utils.py:1676-1680``):

        d gam = [ int dc X^2 - int dg dX^2 - gam int df X^2 ] / int f X^2,   (dg, dc, df) = (g, c, f)_pert - (g, c, f)_base

    with the perturbed coefficients from K1 on the SAME field lines.  Cost per degree of freedom: ``ns`` field lines of
    geometry + one K4 contraction, instead of a full (alpha, theta0) scan + refinement."""
    dev = tables0.tab_mn.device
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    h = engine.grid_spacing(theta_np)
    a = torch.as_tensor(np.asarray(alpha_star, dtype=np.float64)).reshape(-1, 1).to(dev)
    t0 = torch.as_tensor(np.asarray(theta0_star, dtype=np.float64)).reshape(-1).to(dev)
    geo0 = engine.geometry_batch(tables0, a, theta_np)
    sol = engine.solve_base_batch(geo0.base, geo0.dPdrho, t0, h, nth0=1, want_dX=True, want_matrix=False)
    g0, c0, f0 = _gcf_exact(geo0, t0)
    dg, dc, df = [], [], []
    for tp in tables_pert:
        gi, ci, fi = _gcf_exact(engine.geometry_batch(tp, a, theta_np), t0)
        dg.append(gi - g0); dc.append(ci - c0); df.append(fi - f0)
    if not dg:
        return GammaSensitivity(sol.lam.cpu().numpy(), np.zeros((0, t0.numel())), sol.X.cpu().numpy())
    grad = engine.adjoint_batch(sol.lam, sol.X, sol.dX, f0, torch.stack(dg, 1), torch.stack(dc, 1), torch.stack(df, 1))
    return GammaSensitivity(sol.lam.cpu().numpy(), grad.t().contiguous().cpu().numpy(), sol.X.cpu().numpy())


@dataclasses.dataclass
class TableGradient:
    gamma: np.ndarray          # (ns,) growth rate at (alpha*, theta0*)
    grad_mn: torch.Tensor      # (ns, 6, mnmax)      d gamma / d tab_mn
    grad_nyq: torch.Tensor     # (ns, 7, mnmax_nyq)  d gamma / d tab_nyq
    grad_scal: Optional[torch.Tensor] = None    # (ns, 8)  d gamma / d scal (table_gradient(..., scalars=True))
    grad_glob: Optional[torch.Tensor] = None    # (ns, 2)  d gamma / d (phiedge, Aminor_p)

    def predict(self, tables0: engine.DeviceTables, tables_pert) -> np.ndarray:
        """First-order change of every surface's growth rate for each perturbed table set: ``(ndof, ns)``.  With the scalar
        gradients present the changes of ``scal``, ``phiedge`` and ``Aminor_p`` count too; without them they are ignored."""
        return _predict(self, tables0, tables_pert)


def _predict(g, tables0: engine.DeviceTables, tables_pert) -> np.ndarray:
    """Dot products of the table (and, when present, scalar) gradients of ``g`` with each perturbation: ``(ndof, ns)``."""
    out = []
    for tp in tables_pert:
        d = ((tp.tab_mn - tables0.tab_mn) * g.grad_mn).sum(dim=(1, 2)) + ((tp.tab_nyq - tables0.tab_nyq) * g.grad_nyq).sum(dim=(1, 2))
        if g.grad_scal is not None:
            d = (d + ((tp.scal - tables0.scal) * g.grad_scal).sum(1) + (tp.phiedge - tables0.phiedge) * g.grad_glob[:, 0]
                 + (tp.Aminor_p - tables0.Aminor_p) * g.grad_glob[:, 1])
        out.append(d.cpu().numpy())
    return np.array(out).reshape(len(out), -1)


def table_gradient(tables0: engine.DeviceTables, alpha_star, theta0_star, theta, scalars: bool = False) -> TableGradient:
    """SURVEY.md section 8 row f3: the gradient of every surface's maximum growth rate with respect to EVERY Fourier table
    coefficient of its surface, from one eigen-solve per surface -- reverse mode through K1 (``ibs_geometry_adjoint``): K1 on
    the arg-max line -> K2/K3 -> per-point Hellmann-Feynman sensitivities (K4, ``utils.py:1676-1680``) -> adjoint of the
    geometry.  The ``ndofs`` perturbed-equilibrium scans of ``sims_runner_NCSX.py:245-262`` become ``ndofs`` dot products
    (``TableGradient.predict``); ``hellmann_feynman_gamma`` (one K1 per DOF) is the finite-perturbation form of the same.
    ``scalars=True`` (``ibs_geometry_adjoint_scal``) adds the gradient with respect to the surface scalars (iota, iota', p',
    shat, s) and to phiedge / Aminor_p: needed whenever a degree of freedom moves iota, the pressure or phiedge."""
    dev = tables0.tab_mn.device
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    h = engine.grid_spacing(theta_np)
    a = torch.as_tensor(np.asarray(alpha_star, dtype=np.float64)).reshape(-1, 1).to(dev)
    t0 = torch.as_tensor(np.asarray(theta0_star, dtype=np.float64)).reshape(-1).to(dev)
    geo = engine.geometry_batch(tables0, a, theta_np)
    sol = engine.solve_base_batch(geo.base, geo.dPdrho, t0, h, nth0=1, want_dX=True, want_matrix=False, want_gcf=True)
    sg, sc, sf = engine.adjoint_sensitivities(sol.lam, sol.X, sol.dX, sol.f)
    dP = geo.dPdrho.reshape(-1)
    Q = (sc * sol.c).sum(dim=1) / (-dP)
    grads = engine.geometry_adjoint(tables0, a.reshape(-1), theta_np, t0, dP, sg, sc, sf, Q, want_scalars=scalars)
    return TableGradient(sol.lam.cpu().numpy(), *grads)


# ---------------------------------------------------------------------------------------------
# Marginal stability for an optimiser: refined per-surface minimum of kappa* and its gradient with respect to the equilibrium
# ---------------------------------------------------------------------------------------------
def refine_marginal(tables: engine.DeviceTables, alpha_guess, theta0_guess, theta, maxiter: int = 30, ftol: float = 5.0e-11,
                    gtol: float = 2.0e-08, kappa_max: float = 1e3, rtol: float = 1e-12, max_rounds: int = 200, sync_every: int = 4,
                    bounds=((0.0, float(np.pi)), (0.0, 0.5 * float(np.pi)))) -> RefineResult:
    """Refinement of every surface's coarse minimum of kappa* (``marginal_scan``'s ``alpha_crit``, ``theta0_crit``): minimise
    kappa*(alpha, theta0) per surface over the box ``bounds`` -- the ranges of the coarse grid the guesses come from (the
    default is the reference's grid, alpha in [0, pi], theta0 in [0, pi/2]).  The method and the options are those of
    ``refine_maxima(alpha_derivative="exact")``: the batched projected quasi-Newton method of ``csrc/ibs_refine_core.cuh``,
    one round = K1 and its alpha-tangent on one line per surface (``engine.geometry_tangent_batch``) + ``engine.
    marginal_tangent_batch`` (value kappa*, gradient (d kappa*/d alpha, d kappa*/d theta0)) + ``ibs_refine_step``.

    A trial point stable up to ``kappa_max`` (kappa* = +inf) is not usable and the line search backtracks from it.  A surface
    whose starting kappa* is not finite is not refined: it keeps its start and its value there (``success`` False).
    ``fun`` is kappa* at the result."""
    dev = tables.tab_mn.device
    ns = tables.ns
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    theta_d = torch.from_numpy(theta_np).to(dev)
    h = engine.grid_spacing(theta_np)
    as_dev = lambda a: (a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a, dtype=np.float64))).to(dev).reshape(ns)
    st = engine.RefineState(as_dev(alpha_guess), as_dev(theta0_guess), bounds=bounds)
    rounds = 0
    k_start = None
    while rounds < max_rounds:
        for _ in range(sync_every):
            geo = engine.geometry_tangent_batch(tables, st.alphas3[:, 1:2], theta_d)
            m = engine.marginal_tangent_batch(geo.base, geo.dbase, geo.dPdrho, geo.ddPdrho, st.theta0, h, nth0=1, kappa_max=kappa_max,
                                              rtol=rtol)
            if k_start is None:
                k_start = m.kappa.clone()          # the first round evaluates every starting point
            st.step(m.kappa, m.grad, m.info, ftol, gtol, maxiter)
            rounds += 1
        if int(st.nactive.item()) == 0:
            break
    S = st.state.cpu().numpy()
    why = S[:, 19].astype(int)
    unrefined = why == 5                           # failed at the start: kappa* not finite (or the solve flagged it) there
    fun = np.where(unrefined, k_start.cpu().numpy(), S[:, 2])
    return RefineResult(alpha=S[:, 0].copy(), theta0=S[:, 1].copy(), fun=fun, nit=S[:, 20].astype(int), nfev=S[:, 21].astype(int),
                        success=np.isin(why, (1, 2, 3, 4)), nbatches=rounds)


@dataclasses.dataclass
class MarginalGradient:
    kappa: np.ndarray          # (ns,) kappa* at (alpha*, theta0*)
    finite: np.ndarray         # (ns,) bool: kappa* finite (the other rows of the gradients are 0)
    grad_mn: torch.Tensor      # (ns, 6, mnmax)      d kappa* / d tab_mn
    grad_nyq: torch.Tensor     # (ns, 7, mnmax_nyq)  d kappa* / d tab_nyq
    grad_scal: Optional[torch.Tensor] = None    # (ns, 8)  d kappa* / d scal (marginal_gradient(..., scalars=True))
    grad_glob: Optional[torch.Tensor] = None    # (ns, 2)  d kappa* / d (phiedge, Aminor_p)

    def predict(self, tables0: engine.DeviceTables, tables_pert) -> np.ndarray:
        """First-order change of every surface's kappa* for each perturbed table set: ``(ndof, ns)`` (as
        ``TableGradient.predict``)."""
        return _predict(self, tables0, tables_pert)


def marginal_gradient(tables0: engine.DeviceTables, alpha_star, theta0_star, theta, scalars: bool = False, kappa_max: float = 1e3,
                      rtol: float = 1e-12) -> MarginalGradient:
    """Gradient of every surface's kappa* at (alpha*, theta0*) with respect to every Fourier table coefficient (and with
    ``scalars=True`` the surface scalars and phiedge / Aminor_p): one kappa* solve per surface and one reverse-mode pass
    through K1, with no adjoint code of its own.

    kappa* scales as kappa*(t p') = kappa*(p') / t.  So on the tables T_kappa, whose p' (``scal[:, 3]``) is multiplied by each
    surface's kappa*, K1 gives exactly the kappa*-scaled base arrays, and ``ibs_geometry_adjoint_scal`` fed with the per-point
    sensitivities of kappa* (``engine.marginal_sensitivities``, with f not entering) returns d kappa* / d T_kappa.  Its p'
    column multiplied by kappa* is d kappa* / d p'; every other column is d kappa* / dT as it stands.

    At a refined interior minimum (``refine_marginal``) the minimum is stationary in (alpha, theta0), so this is the gradient of
    the surface's refined ``kappa_min`` itself (envelope theorem).  At an unrefined grid point it is the gradient of kappa* at
    that fixed (alpha, theta0).  Rows of surfaces whose kappa* is not finite (stable up to ``kappa_max``, bad input) are 0."""
    dev = tables0.tab_mn.device
    theta_np = theta.cpu().numpy() if isinstance(theta, torch.Tensor) else np.asarray(theta, dtype=np.float64)
    h = engine.grid_spacing(theta_np)
    a = torch.as_tensor(np.asarray(alpha_star, dtype=np.float64)).reshape(-1, 1).to(dev)
    t0 = torch.as_tensor(np.asarray(theta0_star, dtype=np.float64)).reshape(-1).to(dev)
    geo = engine.geometry_batch(tables0, a, theta_np)
    m = engine.marginal_batch(geo.base, geo.dPdrho, t0, h, nth0=1, kappa_max=kappa_max, rtol=rtol, want_X=True)
    fin = (m.kappa > 0) & (m.kappa < float("inf"))
    ks = torch.where(fin, m.kappa, torch.ones_like(m.kappa))
    scal_k = tables0.scal.clone()
    scal_k[:, 3] *= ks
    tk = dataclasses.replace(tables0, scal=scal_k)
    geo_k = engine.geometry_batch(tk, a, theta_np)
    c_k = _gcf_exact(geo_k, t0)[1]
    dk_dg, dk_dc = engine.marginal_sensitivities(geo.base, geo.dPdrho, t0, h, m.kappa, m.X, nth0=1)
    dk_dg = torch.where(fin[:, None], dk_dg, 0.0)
    dk_dc = torch.where(fin[:, None], dk_dc, 0.0)
    dPk = geo_k.dPdrho.reshape(-1)
    Q = torch.where(fin, (dk_dc * c_k).sum(dim=1) / (-dPk), 0.0)
    grads = engine.geometry_adjoint(tk, a.reshape(-1), theta_np, t0, dPk, dk_dg, dk_dc, torch.zeros_like(dk_dg), Q, want_scalars=scalars)
    grads = [torch.where(fin.reshape((-1,) + (1,) * (g.dim() - 1)), g, 0.0) for g in grads]
    if scalars:
        grads[2][:, 3] *= ks
    return MarginalGradient(m.kappa.cpu().numpy(), fin.cpu().numpy(), *grads)


def save_results(path: str, dof_idx: int, iter0: int, result: BallScanResult) -> None:
    """Append one row per call to ``ball_gam<dof>.npy``, ``ball_theta0<dof>.npy``, ``ball_alpha<dof>.npy`` with the
    reference's semantics (``ball_scan.py:359-384``): at ``iter0 == 0`` the placeholder first element written by
    ``arr_create2.py`` is dropped, afterwards rows are stacked."""
    import os
    for name, row in (("ball_gam", result.gamma), ("ball_theta0", result.theta0), ("ball_alpha", result.alpha)):
        fn = os.path.join(path, "%s%d.npy" % (name, int(dof_idx)))
        old = np.load(fn, allow_pickle=True)
        if iter0 == 0:
            new = np.delete(np.append(old, row), 0)
        else:
            new = np.vstack((old, row))
        np.save(fn, new)
