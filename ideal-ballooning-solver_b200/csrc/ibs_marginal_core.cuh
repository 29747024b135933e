// Marginal ballooning stability: the per-lane arithmetic (host/device code).
//
// kappa* of a (field line, theta0) is the critical factor of the pressure gradient at fixed geometry.  K1 puts p' only into
// cvdrift - gbdrift (= -K dpds / B^2) and into dPdrho = -1/2 mean((cvdrift - gbdrift) bmag^2), so scaling p' by kappa is, on
// the base arrays,  cvdrift_k = gbdrift + kappa (cvdrift - gbdrift),  dPdrho_k = kappa dPdrho:  g and f do not move and
//     c(kappa) = kappa c1 + kappa^2 c2,   c1 = -dPdrho (gbdrift + theta0 cvdrift0) / (|gradpar| bmag),
//                                         c2 = -dPdrho (cvdrift - gbdrift) / (|gradpar| bmag).
//     kappa* = inf { kappa > 0 : the discrete pencil has an eigenvalue > 0 }   (the first kappa with count_above(0) >= 1).
// At lam = 0 the count depends on K = D g D + diag(c) alone (Sylvester), so f enters only the optional outputs.  For K1
// output c2 >= 0 pointwise, lam_max(kappa) is convex, lam_max(0) < 0, and the crossing is unique: the count at a trial kappa
// says on which side of kappa* it lies.  Base arrays with c2 < 0 somewhere (e.g. the s-alpha model) are flagged NOT_CONVEX:
// the crossing found is then not certified to be the first one.
//
// Rows are those of the scan solver (ibs_scan_core.cuh, raw_record): scaled by 2 h^2, a_j = g_{j-1} + g_j = 2 gh of the half
// cell, row j of K: a_{j+1} (x_{j+1} - x_j) - a_j (x_j - x_{j-1}) + C_j x_j with C = 2 h^2 c.  A record of a point holds
//     G0 G1 G2 (g = G0 + th0 G1 + th0^2 G2) | Cg C1 Cd  (C = kappa (Cg + th0 C1) + kappa^2 Cd).
//
// One sweep at (kappa, lam = 0) runs the division-free shooting recurrence of the scan solver's forward chain from the left
// Dirichlet end, X_j = a_j X_{j-1} + W_{j-1}, W_j = a_j W_{j-1} - C_j X_j (state scaled by the running product of the a).  With
// D_j the leading principal minors of K, X_{j+1} ~ (-1)^j D_j, so the LDL^T pivot p_j = D_j / D_{j-1} is positive exactly where
// X changes sign between rows j and j+1: count(0) = sign changes of X_1 .. X_{N-1} (the node count of the solver, with its
// sign-bit rule: an exact zero counts as +0, i.e. a zero pivot as a non-positive one).  det K ~ X_{N-1} (the a do not depend
// on kappa), so the kappa-tangent (X', W') of the same recurrence gives phi = d log|det K| / d kappa = X'_{N-1} / X_{N-1}
// = sum_j p_j' / p_j without a division per row, and the Newton step on the determinant is kappa - 1 / phi.
//
// The optional outputs come from the null vector x* of K(kappa*), one twisted factorisation: forward pivots (kept in the
// caller's X row as scratch), backward pivots, the twist row k = argmin |p_k + q_k - d_k|, then x from row k outwards.
//
// The first-order response of kappa* at x* (point_forms, point_sensitivities) gives d kappa* / d alpha from the records'
// alpha-tangent and the per-point sensitivities d kappa* / d g_j, d kappa* / d c_j that the reverse mode of K1 consumes.
#pragma once
#include <cmath>
#include <cstdint>

#include "../../include/ibs_b200.h"
#include "ibs_scan_core.cuh"

namespace ibs {
namespace marg {
using scan::Rec;
using scan::exp_max2;
using scan::not_finite;
using scan::not_pos_normal;
using scan::pow2;
using scan::raw_record;
using scan::sign_bit;

constexpr int MREC = 6;                 // doubles per record: G0 G1 G2 Cg C1 Cd
constexpr int MAXSWEEP = 96;            // sweeps per solve before giving up (NOT_CONVERGED)
constexpr int CHAIN = 4;                // consecutive solves of one lane; a solve starts from its predecessor's kappa* on the same line
constexpr int RESCALE = 16;             // rows between rescalings of the shooting state
constexpr double GROW = 8.0;            // largest factor by which one step may move kappa up before a crossing is found
constexpr int FLAG_NOT_CONVERGED = 1, FLAG_BAD_INPUT = 2, FLAG_STABLE_TO_KMAX = 8, FLAG_NOT_CONVEX = 16;   // = IBS_FLAG_*

struct MRec { double G0, G1, G2, Cg, C1, Cd; };

IBS_HD MRec load_mrec(const double* p) {
    MRec r;
#if defined(__CUDA_ARCH__)
    const double2* q = reinterpret_cast<const double2*>(p);          // 48-byte records, 16-byte aligned
    const double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    r.G0 = a.x; r.G1 = a.y; r.G2 = b.x; r.Cg = b.y; r.C1 = c.x; r.Cd = c.y;
#else
    r.G0 = p[0]; r.G1 = p[1]; r.G2 = p[2]; r.Cg = p[3]; r.C1 = p[4]; r.Cd = p[5];
#endif
    return r;
}

// Record of one point from its eight base values (IBS_BASE_* order) -- the scan solver's raw_record, evaluated once with
// gbdrift and once with cvdrift - gbdrift in place of cvdrift.  R = 2 h^2 f / g is returned for the optional outputs and the
// input checks; it is not part of the record.
IBS_HD MRec marginal_record(const double* b8, double dP, double h2, double& R) {
    const Rec r = raw_record(b8[0], b8[1], b8[7], b8[3], b8[4], b8[5], b8[6], dP, h2);
    const Rec d = raw_record(b8[0], b8[1], b8[2] - b8[7], 0.0, b8[4], b8[5], b8[6], dP, h2);
    MRec m;
    m.G0 = r.G0; m.G1 = r.G1; m.G2 = r.G2; m.Cg = r.C0; m.C1 = r.C1; m.Cd = d.C0;
    R = r.R;
    return m;
}
// per-line flags of a record: BAD_INPUT (non-finite, or f / g not a positive normal number), NOT_CONVEX (c2 < 0)
IBS_HD int record_flags(const MRec& m, double R) {
    const bool bad = not_finite(m.G0) | not_finite(m.G1) | not_finite(m.G2) | not_finite(m.Cg) | not_finite(m.C1) | not_finite(m.Cd) |
                     not_pos_normal(R);
    return (bad ? FLAG_BAD_INPUT : 0) | (m.Cd < 0.0 ? FLAG_NOT_CONVEX : 0);
}

// record of point j of a line (b: its 8 x N base arrays) into out[MREC]; returns the point's record_flags
IBS_HD int prep_point(const double* b, int N, int j, double dP, double h2, double* out) {
    double b8[IBS_NBASE];
    for (int q = 0; q < IBS_NBASE; ++q) b8[q] = b[(size_t)q * N + j];
    double R;
    const MRec m = marginal_record(b8, dP, h2, R);
    out[0] = m.G0; out[1] = m.G1; out[2] = m.G2; out[3] = m.Cg; out[4] = m.C1; out[5] = m.Cd;
    return record_flags(m, R);
}

IBS_HD double g_of(const MRec& r, double th0) { return fma(th0, fma(th0, r.G2, r.G1), r.G0); }
IBS_HD double c1_of(const MRec& r, double th0) { return fma(th0, r.C1, r.Cg); }

// ---- one sweep at (kappa, lam = 0) ----------------------------------------------------------------------------------------
struct SweepOut { int count; double phi; bool bad; };

template <bool CHECK>
IBS_HD SweepOut sweep(const double* rec, int N, double th0, double kap) {
    double gp = g_of(load_mrec(rec), th0);
    bool bad = CHECK && not_pos_normal(gp);
    double X = 0.0, W = 1.0, Xd = 0.0, Wd = 0.0;          // left Dirichlet end: x = 0, w' = 1; the tangent starts at zero
    unsigned prev = 0;                                    // sign of X_1 = 1 is +
    int count = 0;
    const double* p = rec + MREC;
#pragma unroll 1
    for (int j0 = 1; j0 < N; j0 += RESCALE) {
        const int j1 = scan::imin(N, j0 + RESCALE);
#pragma unroll 4
        for (int j = j0; j < j1; ++j, p += MREC) {
            const MRec r = load_mrec(p);
            const double g = g_of(r, th0);
            const double a = g + gp;
            gp = g;
            const double u = fma(kap, r.Cd, c1_of(r, th0));    // C = kappa u,  dC/dkappa = u + kappa Cd
            const double C = kap * u, Cp = fma(kap, r.Cd, u);
            const double Xn = fma(a, X, W), Xdn = fma(a, Xd, Wd);
            Wd = fma(-Cp, Xn, fma(-C, Xdn, a * Wd));
            W = fma(-C, Xn, a * W);
            X = Xn; Xd = Xdn;
            const unsigned s = sign_bit(X);
            count += (int)(s ^ prev);
            prev = s;
            if (CHECK) bad |= not_pos_normal(g) | not_finite(C);
        }
        const double sc = pow2(-scan::imax(exp_max2(X, W), exp_max2(Xd, Wd)));
        X *= sc; W *= sc; Xd *= sc; Wd *= sc;
    }
    SweepOut o;
    o.count = count;          // (the last sign change, between X_{N-2} and X_{N-1}, is that of the last pivot)
    o.phi = Xd / X;
    o.bad = bad;
    return o;
}

// ---- root finder ----------------------------------------------------------------------------------------------------------
struct RootOut { double kappa; int sweeps, flags; };

// Bracket [lo, hi]: count(0; lo) = 0 (lo = 0 holds without a sweep: c = 0, g > 0), count(0; hi) >= 1.  From k0 a sweep says on
// which side kappa* lies.  Steps are Newton steps on det K(kappa), aimed past the predicted root by its predicted error
// (min(d^2, d / 4) for a step of relative size d, at least rtol / 4), so that the sweeps alternate sides and both ends of the
// bracket close in.  Before the first unstable point a step moves kappa up by at most GROW (doubling where Newton does not
// point up), capped at kappa_max.  Inside the bracket the fall-back is bisection (geometric while lo = 0): where two or more
// eigenvalues are above 0 (the nearest root of det K is then another crossing), where the Newton step leaves the bracket, and
// where it is not below half the step before the last one (the safeguard of rtsafe).  Stops when hi - lo <= rtol hi and
// returns hi: the smallest kappa certified unstable.
IBS_HD RootOut find_root(const double* rec, int N, double th0, double k0, double kmax, double rtol) {
    const double inf = INFINITY;
    RootOut o; o.kappa = inf; o.sweeps = 0; o.flags = 0;
    double lo = 0.0, hi = inf, dx = inf, dxold = inf;
    double k = fmin(k0, kmax);
    for (;;) {
        const SweepOut s = (o.sweeps == 0) ? sweep<true>(rec, N, th0, k) : sweep<false>(rec, N, th0, k);
        ++o.sweeps;
        if (s.bad) { o.kappa = NAN; o.flags = FLAG_BAD_INPUT; return o; }
        const bool up = s.count >= 1;
        if (up) hi = k; else lo = k;
        if (hi < inf && hi - lo <= rtol * hi) break;
        if (!up && k >= kmax) { o.flags = FLAG_STABLE_TO_KMAX; return o; }
        if (o.sweeps >= MAXSWEEP) { o.flags = FLAG_NOT_CONVERGED; break; }
        double cand = k - 1.0 / s.phi;
        const double d = fabs(k - cand) / k, aim = fmax(0.25 * rtol, fmin(d * d, 0.25 * d));
        cand *= up ? 1.0 - aim : 1.0 + aim;
        double next;
        if (hi == inf) {
            next = (cand > k && cand < GROW * k) ? cand : ((cand >= GROW * k) ? GROW * k : 2.0 * k);
            next = fmin(next, kmax);
        } else {
            const bool newton = s.count <= 1 && cand > lo && cand < hi && fabs(cand - k) <= 0.5 * dxold;
            next = newton ? cand : (lo > 0.0 ? 0.5 * (lo + hi) : 0.5 * hi);
        }
        dxold = dx; dx = fabs(next - k);
        k = next;
    }
    o.kappa = hi;
    return o;
}

// ---- optional outputs: the null vector at kappa* and the two derivatives --------------------------------------------------
struct Derivs { double dlam_dkappa, dkappa_dtheta0; };

// diagonal d_j and the coupling a_{j+1} to the next row of row j at kappa, from the records of rows j-1, j, j+1
IBS_HD void row_diag(const MRec& rm, const MRec& r0, const MRec& rp, double th0, double kap, double& d, double& a_lo, double& a_hi) {
    const double gm = g_of(rm, th0), g0 = g_of(r0, th0), gq = g_of(rp, th0);
    a_lo = gm + g0; a_hi = g0 + gq;
    d = -(a_lo + a_hi) + kap * fma(kap, r0.Cd, c1_of(r0, th0));
}

// x* >= 0 with max 1 into X[0..N-1] (X doubles as the pivot scratch); b: the line's base arrays (8 x N), read for f.  Returns the
// derivatives  dlam/dkappa = x^T dK/dkappa x / x^T F x  and  dkappa*/dtheta0 = -x^T dK/dtheta0 x / x^T dK/dkappa x.
IBS_HD Derivs null_vector(const double* rec, const double* b, int N, double h2, double th0, double kap, double* X) {
    const int M = N - 2;
    auto R = [&](int j) -> MRec { return load_mrec(rec + (size_t)j * MREC); };
    const double tiny = 2.2250738585072014e-308;
    // forward pivots p_j -> X[j]
    {
        double p = 0.0, aprev = 0.0;
        MRec rm = R(0), r0 = R(1);
        for (int j = 1; j <= M; ++j) {
            const MRec rp = R(j + 1);
            double d, alo, ahi;
            row_diag(rm, r0, rp, th0, kap, d, alo, ahi);
            p = (j == 1) ? d : d - aprev * aprev / p;
            if (p == 0.0) p = -tiny;
            X[j] = p;
            aprev = ahi;
            rm = r0; r0 = rp;
        }
    }
    // backward pivots q_j, twist row k = argmin |p_j + q_j - d_j|
    int k = 1;
    {
        double q = 0.0, anext = 0.0, best = INFINITY;
        MRec rp = R(N - 1), r0 = R(M);
        for (int j = M; j >= 1; --j) {
            const MRec rm = R(j - 1);
            double d, alo, ahi;
            row_diag(rm, r0, rp, th0, kap, d, alo, ahi);
            q = (j == M) ? d : d - anext * anext / q;
            if (q == 0.0) q = -tiny;
            const double gam = fabs(X[j] + q - d);
            if (gam < best) { best = gam; k = j; }
            anext = alo;
            rp = r0; r0 = rm;
        }
    }
    // backward pivots again, kept for the rows below the twist: X[j] = q_j for j > k
    {
        double q = 0.0, anext = 0.0;
        MRec rp = R(N - 1), r0 = R(M);
        for (int j = M; j > k; --j) {
            const MRec rm = R(j - 1);
            double d, alo, ahi;
            row_diag(rm, r0, rp, th0, kap, d, alo, ahi);
            q = (j == M) ? d : d - anext * anext / q;
            if (q == 0.0) q = -tiny;
            X[j] = q;
            anext = alo;
            rp = r0; r0 = rm;
        }
    }
    // x from the twist row outwards: x_j = -a_{j+1} x_{j+1} / p_j above it, x_j = -a_j x_{j-1} / q_j below it
    double xmax = 1.0;
    {
        double x = 1.0;
        for (int j = k - 1; j >= 1; --j) {
            const double a = g_of(R(j), th0) + g_of(R(j + 1), th0);
            x = -a * x / X[j];
            X[j] = x;
            if (fabs(x) > fabs(xmax)) xmax = x;
        }
        X[k] = 1.0;
        x = 1.0;
        for (int j = k + 1; j <= M; ++j) {
            const double a = g_of(R(j - 1), th0) + g_of(R(j), th0);
            x = -a * x / X[j];
            X[j] = x;
            if (fabs(x) > fabs(xmax)) xmax = x;
        }
        X[0] = 0.0; X[N - 1] = 0.0;
    }
    // normalise (max 1; the nodeless ground state is then >= 0) and form the three quadratic forms
    const double s = 1.0 / xmax;
    double qk = 0.0, qf = 0.0, qt = 0.0;
    double xprev = 0.0, gdprev = fma(2.0 * th0, R(0).G2, R(0).G1);
    for (int j = 1; j < N; ++j) {
        const MRec r = R(j);
        const double x = X[j] * s;
        X[j] = x;
        const double gd = fma(2.0 * th0, r.G2, r.G1), dx = x - xprev;
        qt = fma(-(gd + gdprev), dx * dx, qt);                   // -a'_j (x_j - x_{j-1})^2 over the half cells 1 .. N-1
        if (j <= M) {
            const double Rj = raw_record(b[(size_t)IBS_BASE_BMAG * N + j], b[(size_t)IBS_BASE_GRADPAR * N + j], 0.0, 0.0, 0.0, 0.0,
                                         0.0, 0.0, h2).R;           // f = g R
            const double x2 = x * x;
            qk = fma(fma(2.0 * kap, r.Cd, c1_of(r, th0)), x2, qk);
            qf = fma(g_of(r, th0) * Rj, x2, qf);
            qt = fma(kap * r.C1, x2, qt);
        }
        xprev = x; gdprev = gd;
    }
    Derivs o;
    o.dlam_dkappa = qk / qf;
    o.dkappa_dtheta0 = -qt / qk;
    return o;
}

// ---- first-order response of kappa* at the null vector: alpha-tangent and per-point sensitivities ------------------------
// For any quantity q that K depends on, d kappa* / dq = -x^T (dK/dq) x / qk with qk = x^T (dK/dkappa) x.  With the rows of
// K as above, x^T K x = -sum_cells a_j (x_j - x_{j-1})^2 + sum_j C_j x_j^2, so point j enters through its g (the cells j and
// j+1 that exist) and through its C (interior points only).  These terms are summed per point; the caller adds them up.

// alpha-tangent of a point's record along (d8, ddP): the chain rule through marginal_record / raw_record
IBS_HD MRec record_tangent(const double* b8, const double* d8, double dP, double ddP, double h2) {
    const double B = b8[IBS_BASE_BMAG], dB = d8[IBS_BASE_BMAG];
    const double gp = fabs(b8[IBS_BASE_GRADPAR]), dgp = (b8[IBS_BASE_GRADPAR] < 0.0 ? -1.0 : 1.0) * d8[IBS_BASE_GRADPAR];
    const double gpB = gp * B, gpoB = gp / B, mdP = -2.0 * h2 * dP / gpB;
    const double d_gpoB = (dgp - gpoB * dB) / B;                                  // d (gp / B)
    const double d_mdP = -2.0 * h2 * ddP / gpB - mdP * (dgp / gp + dB / B);       // d (-2 h^2 dP / (gp B))
    const double gb = b8[IBS_BASE_GBDRIFT], dgb = d8[IBS_BASE_GBDRIFT];
    MRec t;
    t.G0 = d_gpoB * b8[IBS_BASE_GDS2] + gpoB * d8[IBS_BASE_GDS2];
    t.G1 = 2.0 * (d_gpoB * b8[IBS_BASE_GDS21] + gpoB * d8[IBS_BASE_GDS21]);
    t.G2 = d_gpoB * b8[IBS_BASE_GDS22] + gpoB * d8[IBS_BASE_GDS22];
    t.Cg = d_mdP * gb + mdP * dgb;
    t.C1 = d_mdP * b8[IBS_BASE_CVDRIFT0] + mdP * d8[IBS_BASE_CVDRIFT0];
    t.Cd = d_mdP * (b8[IBS_BASE_CVDRIFT] - gb) + mdP * (d8[IBS_BASE_CVDRIFT] - dgb);
    return t;
}

// (x_j - x_{j-1})^2 + (x_{j+1} - x_j)^2 over the cells of point j that exist (x: the solve's N values)
IBS_HD double cell_weight(const double* x, int N, int j) {
    double w = 0.0;
    if (j > 0) { const double d = x[j] - x[j - 1]; w = d * d; }
    if (j < N - 1) { const double d = x[j + 1] - x[j]; w = fma(d, d, w); }
    return w;
}

struct PointForms { double qk, qa; };

// point j's share of qk = x^T dK/dkappa x and of qa = x^T dK/dalpha x.  b, db: the line's 8 x N base arrays and their alpha-
// tangent (db = null: qk only); dP, ddP: dPdrho and its tangent.
IBS_HD PointForms point_forms(const double* b, const double* db, int N, int j, double dP, double ddP, double h2, double th0, double kap,
                              const double* x) {
    double b8[IBS_NBASE];
    for (int q = 0; q < IBS_NBASE; ++q) b8[q] = b[(size_t)q * N + j];
    double R;
    const MRec m = marginal_record(b8, dP, h2, R);
    const bool inner = j > 0 && j < N - 1;
    const double x2 = inner ? x[j] * x[j] : 0.0;
    PointForms o;
    o.qk = fma(2.0 * kap, m.Cd, c1_of(m, th0)) * x2;
    o.qa = 0.0;
    if (db) {
        double d8[IBS_NBASE];
        for (int q = 0; q < IBS_NBASE; ++q) d8[q] = db[(size_t)q * N + j];
        const MRec t = record_tangent(b8, d8, dP, ddP, h2);
        o.qa = fma(kap * fma(kap, t.Cd, c1_of(t, th0)), x2, -g_of(t, th0) * cell_weight(x, N, j));
    }
    return o;
}

// per-point sensitivities of kappa* in the reference's unscaled coefficients (utils.py:1560-1562) at kappa*:
//   d kappa* / d g_j = cell_weight_j / qk,   d kappa* / d c_j = -2 h^2 x_j^2 / qk (0 at the Dirichlet ends)
IBS_HD void point_sensitivities(const double* x, int N, int j, double h2, double inv_qk, double& dk_dg, double& dk_dc) {
    dk_dg = cell_weight(x, N, j) * inv_qk;
    dk_dc = (j > 0 && j < N - 1) ? -2.0 * h2 * x[j] * x[j] * inv_qk : 0.0;
}

// ---- one lane: CHAIN consecutive solves ----------------------------------------------------------------------------------
struct MarginalArgs {
    const double* rec;           // [nline][N][MREC], or [nsolve][N][MREC] (the record block of each solve's line) if rec_per_solve
    const double* base;          // [nline][8][N]
    const double* dPdrho;        // [nline]
    const int* line_flags;       // [nline] (or [nsolve], as rec): record_flags of the line, or-ed over its points
    const double* theta0;        // [nsolve]
    const int* line_of_solve;    // [nsolve] or null: line = s / nth0
    int nth0, nsolve, N;
    bool rec_per_solve;
    double h2, kmax, rtol;
    double* kappa;               // [nsolve]
    double* dlam_dkappa;         // [nsolve] or null
    double* dkappa_dtheta0;      // [nsolve] or null
    double* X;                   // [nsolve][N] or null (also the pivot scratch of the derivatives)
    int* info;                   // [nsolve] or null: sweeps | flags << 16
};

// A solve starts at kappa = 1 (the pressure profile as given), or at its predecessor's kappa* when that is a finite value on
// the same line: kappa* is smooth in theta0.  The chains are fixed runs of CHAIN solves, so a solve's start (and with it every
// bit of its result) does not depend on how the batch was given: scan-shaped and line_of_solve batches agree.
IBS_HD void solve_chain(const MarginalArgs& A, int chain) {
    const int s0 = chain * CHAIN, s1 = scan::imin(A.nsolve, s0 + CHAIN);
    int prev_line = -1;
    double prev_kappa = NAN;
    for (int s = s0; s < s1; ++s) {
        const int line = A.line_of_solve ? A.line_of_solve[s] : s / A.nth0;
        const double* rec = A.rec + (size_t)(A.rec_per_solve ? s : line) * A.N * MREC;
        const double th0 = A.theta0[s], dP = A.dPdrho[line];
        const int lf = A.line_flags[A.rec_per_solve ? s : line];
        const double k0 = (line == prev_line && prev_kappa > 0.0 && prev_kappa < INFINITY) ? prev_kappa : 1.0;
        RootOut r;
        if (lf & FLAG_BAD_INPUT) { r.kappa = NAN; r.sweeps = 0; r.flags = FLAG_BAD_INPUT; }
        else if (dP == 0.0) { r.kappa = INFINITY; r.sweeps = 0; r.flags = FLAG_STABLE_TO_KMAX; }     // c = 0: never unstable
        else r = find_root(rec, A.N, th0, k0, A.kmax, A.rtol);
        r.flags |= lf & FLAG_NOT_CONVEX;
        A.kappa[s] = r.kappa;
        if (A.info) A.info[s] = r.sweeps | (r.flags << 16);
        const bool fin = r.kappa > 0.0 && r.kappa < INFINITY;
        if (A.X) {
            double* Xs = A.X + (size_t)s * A.N;
            Derivs d;
            if (fin) d = null_vector(rec, A.base + (size_t)line * IBS_NBASE * A.N, A.N, A.h2, th0, r.kappa, Xs);
            else {
                for (int j = 0; j < A.N; ++j) Xs[j] = NAN;
                d.dlam_dkappa = NAN; d.dkappa_dtheta0 = NAN;
            }
            if (A.dlam_dkappa) A.dlam_dkappa[s] = d.dlam_dkappa;
            if (A.dkappa_dtheta0) A.dkappa_dtheta0[s] = d.dkappa_dtheta0;
        }
        prev_line = line; prev_kappa = r.kappa;
    }
}

}  // namespace marg
}  // namespace ibs
