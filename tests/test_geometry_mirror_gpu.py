"""K1's mirror fold on axisymmetric tables: residues r and (c - r) mod P of a grid symmetric about theta = 0 (modulo one
poloidal turn) share one Newton solve and one set of mode sums.  The folded evaluation must agree with the point-by-point
one (IBS_GEO_FOLD=0) to rounding, with the tolerances of the periodicity fold, and the fold that ran is identified from the
bits of theta_vmec."""
import numpy as np
import pytest

from test_geometry_gpu import _d3d_tables, _geometry_with_fold

pytestmark = pytest.mark.gpu

H = 2 * np.pi / 256
T = 128                         # units per chunk (GEO_THREADS)


def _period_and_mirror(theta):
    """The kernel's candidates: P = rint(2 pi / h), c from theta[0] and h."""
    h = theta[1] - theta[0]
    P = int(np.rint(2 * np.pi / h))
    cr = -2.0 * theta[0] / h
    cr -= P * np.floor(cr / P)
    return P, int(np.rint(cr)) % P


def _chunk_split(ns, units, grid):
    """The kernel's work split: CTA b takes units [W b / G, W (b + 1) / G) of W = ns * units and runs them in chunks of T,
    a chunk ending at the latest at the second surface boundary.  Returns (chunks straddling a surface boundary, chunks cut
    short at the second boundary)."""
    W, straddle, cut = ns * units, 0, 0
    for b in range(grid):
        u0, ue = W * b // grid, W * (b + 1) // grid
        while u0 < ue:
            js0 = u0 // units
            u1 = min(u0 + T, ue, (js0 + 2) * units)
            straddle += (u1 - 1) // units != js0
            cut += u1 < min(u0 + T, ue)
            u0 = u1
    return straddle, cut


def _periodic_bits(tv, theta, P):
    """theta_vmec[j] = theta_vmec[j mod P] + (theta[j] - theta[j mod P]) bit for bit: what the periodicity fold writes."""
    r = np.arange(len(theta)) % P
    return tv == tv[:, r] + (theta - theta[r])


def _mirror_bits(tv, theta, P, c):
    """What the mirror fold writes: the representative r of every orbit (r <= (c - r) mod P) by the periodicity fold, every
    point j of its mirror residue as (theta[j] + theta[r]) - theta_vmec[r]."""
    res = np.arange(len(theta)) % P
    mir = (c - res) % P
    rep = np.where(res <= mir, res, mir)
    fold = tv[:, rep] + (theta - theta[rep])
    mirror = (theta + theta[rep]) - tv[:, rep]
    return tv == np.where(res <= mir, fold, mirror)


@pytest.mark.parametrize("grid,ns,alpha", [
    ("bench_shifted", 5, [0.0, 0.7, 2.9]),     # periodic (P = 256) but not mirror-symmetric: periodicity fold only
    ("odd_period", 5, [0.0, 0.7, 2.9]),        # P = 101, c = 0: one self-mirror residue
    ("odd_mirror", 5, [0.0, 0.7, 2.9]),        # P = 256, c = 255: no self-mirror residue
    ("bench_one_alpha", 80, [0.4]),            # 129 orbits per surface and a full persistent grid: chunks straddle surfaces
    ("short_period", 1300, [0.4]),             # 9 orbits per surface: chunks cut at the second surface boundary
])
def test_axisymmetric_mirror_fold_matches_direct(cuda_lib, monkeypatch, grid, ns, alpha):
    import torch
    st = _d3d_tables(ns)
    if grid == "bench_shifted":
        theta = np.linspace(-4 * np.pi, 4 * np.pi, 1025) + 0.3 * H
    elif grid == "odd_period":
        theta = -3 * np.pi + (2 * np.pi / 101) * np.arange(3 * 101 + 1)
    elif grid == "odd_mirror":
        theta = -4 * np.pi + H / 2 + H * np.arange(1024)
    elif grid == "bench_one_alpha":
        theta = np.linspace(-4 * np.pi, 4 * np.pi, 1025)
    else:
        theta = np.linspace(-2 * np.pi, 2 * np.pi, 33)
    alpha = np.array(alpha)
    P, c = _period_and_mirror(theta)
    if grid in ("bench_one_alpha", "short_period"):
        # the persistent grid is min(surfaces x 128-point tiles, SMs x CTAs / SM); whatever the CTAs / SM (1..4), this
        # case has chunks that straddle surfaces, and on the short period chunks cut short at the second boundary
        orbits = len({min(r, (c - r) % P) for r in range(P)})
        tiles = ns * ((len(alpha) * len(theta) + T - 1) // T)
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        for per_sm in (1, 2, 3, 4):
            straddle, cut = _chunk_split(ns, len(alpha) * orbits, min(tiles, sms * per_sm))
            assert straddle > 0 and (cut > 0 or grid == "bench_one_alpha"), (per_sm, straddle, cut)
    b1, t1, i1, d1 = _geometry_with_fold(st, alpha, theta, True, monkeypatch)
    b0, t0, i0, d0 = _geometry_with_fold(st, alpha, theta, False, monkeypatch)
    assert np.all((i0 >> 16) == 0) and np.all((i1 >> 16) == 0)
    np.testing.assert_allclose(t1, t0, rtol=0, atol=2e-13)
    scale = np.max(np.abs(b0), axis=-1, keepdims=True)
    assert np.max(np.abs(b1 - b0) / scale) < 1e-12
    np.testing.assert_allclose(d1, d0, rtol=1e-12)
    # which fold ran: its bit pattern holds at every point of the folded run, and not at every point of the direct one
    tv1, tv0 = t1.reshape(-1, len(theta)), t0.reshape(-1, len(theta))
    bits = (lambda tv: _periodic_bits(tv, theta, P)) if grid == "bench_shifted" else (lambda tv: _mirror_bits(tv, theta, P, c))
    assert np.all(bits(tv1))
    assert not np.all(bits(tv0))
