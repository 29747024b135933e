// Reverse mode of the field-line geometry: d(lambda) / d(Fourier table coefficient)  (SURVEY.md section 8 row f3).
//
// The reference obtains the Jacobian of the ballooning penalty by finite differences over ndofs + 1 perturbed equilibria,
// each with a full scan (/root/reference/sims_runner_NCSX.py:245-262).  With the eigen-pair of the base equilibrium in hand
// the Hellmann-Feynman formula the reference itself uses for its (alpha, theta0) gradients (utils.py:1676-1680) gives the
// first-order change of lambda for ANY change of the coefficient arrays,
//     d lam = sum_j ( s^g_j dg_j + s^c_j dc_j + s^f_j df_j ),        s^g, s^c, s^f from ibs_adjoint_sensitivities,
// and g, c, f are explicit functions of the 19 mode sums of each point (utils.py:432-720) and of dPdrho (a mean over the line,
// ball_scan.py:262).  This file chains that back to the tables:
//   stage A (one thread per point):  theta_vmec (Newton), the 19 mode sums S_r and their theta_vmec-derivatives; then
//       v_r = d Phi_j / d S_r   with   Phi_j = s^g g - dP s^c chat + s^f f + (Q / 2N) (cvdrift - gbdrift) bmag^2
//       (chat = c / (-dP), Q = sum_j s^c_j chat_j: the dPdrho term folded back onto the points), by FORWARD-mode automatic
//       differentiation of the pointwise algebra (a value + one derivative, 19 sweeps: no hand-derived adjoint to get wrong),
//       and the weight u = -(d Phi / d theta_vmec) / (1 + d lambda / d theta_vmec) of the implicit theta_vmec(l_mn) dependence;
//   stage B (one thread per (surface, mode)):  the transposed mode sum over the points of the line,
//       d lam / d rmnc[mn] = sum_j ( v_R cos a - m v_Rt sin a + n v_Rp sin a ),  a = m theta_vmec - n phi,   etc.
// Gradients are with respect to the per-surface tables tab_mn (6 rows) and tab_nyq (7 rows) at fixed scalars (iota, shat,
// p', iota') and globals (phiedge, Aminor_p).  ibs_geometry_adjoint_scal adds the stage-A instantiation SCAL = true, which
// forms per point only the total d Phi_j / dx of the seven scalars K1 reads -- x = s, iota, iota', p', shat (scal columns
// 0-4), phiedge, Aminor_p -- by seven forward sweeps, and geo_adjoint_scal_sum_kernel sums them over the line in a fixed order
// (deterministic).  The table part is the same two kernels with the same launches as ibs_geometry_adjoint, so its outputs are
// bit-identical (a point kernel doing both the table and the scalar sweeps did not reproduce them bit for bit).  iota also
// moves the field line, phi = phi_c + (theta_p - alpha) / iota, hence the mode sums through a = m theta_vmec - n phi with
//     d S_r / d iota = (P_r + T_r theta_phi) d phi / d iota,   P_r = d S_r / d phi at fixed theta_vmec,
//     theta_phi = d theta_vmec / d phi = -S_Lp / (1 + S_Lt)    (implicit function of the Newton residual).
// Not a hot kernel: ns field lines (each surface's arg-max line), direct mode sums.
#include "ibs_geometry_ad.cuh"

namespace ibs {

constexpr int NSX = 7;    // scalar sweeps: scal columns 0..4 (s, iota, iota', p', shat), phiedge, Aminor_p

// Phi_j as a function of the 19 mode sums (the pointwise algebra of geo_point_epilogue, ibs_geometry.cu, on T = D1)
template <class C>
__device__ D1 phi_point(const D1 (&S)[NSUM], const PointConst<C>& k) {
    D1 o[IBS_NBASE];
    base_point(S, k, o);
    const D1 bmag = o[IBS_BASE_BMAG], gradpar = o[IBS_BASE_GRADPAR], cvdrift = o[IBS_BASE_CVDRIFT], gbdrift0 = o[IBS_BASE_CVDRIFT0];
    const D1 gds2 = o[IBS_BASE_GDS2], gds21 = o[IBS_BASE_GDS21], gds22 = o[IBS_BASE_GDS22], gbdrift = o[IBS_BASE_GBDRIFT];
    // theta0 shift and the coefficients (ball_scan.py:267-268, utils.py:1560-1562)
    const D1 cv_f = cvdrift + D1(k.th0) * gbdrift0;
    const D1 gd_f = gds2 + D1(2.0 * k.th0) * gds21 + D1(k.th0 * k.th0) * gds22;
    const D1 gp = dabs(gradpar);
    const D1 g = gp * gd_f / bmag;
    const D1 chat = cv_f / (gp * bmag);                        // c = -dPdrho chat
    const D1 f = gd_f / (bmag * bmag * bmag * gp);
    return D1(k.sg) * g - D1(k.dP * k.sc) * chat + D1(k.sf) * f + D1(k.qw) * (cvdrift - gbdrift) * bmag * bmag;
}

struct GeoAdjParams {
    const double* tab_mn; const double* tab_nyq; const double* scal;
    const double* xm; const double* xn; const double* xm_nyq; const double* xn_nyq;
    int ns, mnmax, mnmax_nyq, nl;
    const double* alpha; const double* theta; const double* theta0; const double* dPdrho;
    const double* sg; const double* sc; const double* sf; const double* Q;
    double phi_center, psi_e, L_ref;
    double* work;          // [ns][NSUM + 3][nl]: v_r (19), u, theta_vmec, phi
    double* grad_mn; double* grad_nyq;
    double* work_scal;     // [ns][NSX][nl]: d Phi_j / dx of the scalar sweeps (ibs_geometry_adjoint_scal only)
    double* grad_scal; double* grad_glob;      // [ns][IBS_NSCAL], [ns][2]
};

template <bool SCAL>
__global__ void __launch_bounds__(128)
geo_adjoint_point_kernel(const GeoAdjParams p) {
    const long long pt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pt >= (long long)p.ns * p.nl) return;
    const int js = (int)(pt / p.nl), jl = (int)(pt - (long long)js * p.nl);
    const double* sc = p.scal + (size_t)js * IBS_NSCAL;
    PointConst<double> k;
    k.s_val = sc[0]; k.iota = sc[1]; k.d_iota = sc[2]; k.dpds = sc[3]; k.shat = sc[4];
    k.psi_e = p.psi_e; k.L_ref = p.L_ref;
    const double theta_p = p.theta[jl], phi = p.phi_center + (theta_p - p.alpha[js]) / k.iota;
    sincos(phi, &k.sp, &k.cp);
    k.dphi = phi - p.phi_center;
    const size_t o = (size_t)js * p.nl + jl;
    k.th0 = p.theta0[js]; k.dP = p.dPdrho[js]; k.sg = p.sg[o]; k.sc = p.sc[o]; k.sf = p.sf[o]; k.qw = p.Q[js] / (2.0 * p.nl);
    const int mn = p.mnmax, mq = p.mnmax_nyq;
    const double* tm = p.tab_mn + (size_t)js * IBS_TAB_MN_ROWS * mn;
    const double* tq = p.tab_nyq + (size_t)js * IBS_TAB_NYQ_ROWS * mq;
    // theta_vmec (utils.py:391-416), Newton with the analytic derivative
    double th = theta_p;
    for (int it = 0; it < 50; ++it) {
        double f = th - theta_p, d = 1.0;
        for (int q = 0; q < mn; ++q) {
            double sa, ca;
            sincos(p.xm[q] * th - p.xn[q] * phi, &sa, &ca);
            f = fma(tm[2 * mn + q], sa, f);
            d = fma(tm[2 * mn + q] * p.xm[q], ca, d);
        }
        const double dth = f / d;
        th -= dth;
        if (fabs(dth) <= 4.5e-16 * fmax(1.0, fabs(th))) break;
    }
    // the 19 sums and their theta_vmec-derivatives
    double S[NSUM], T[NSUM], P[NSUM];      // P_r = d S_r / d phi at fixed theta_vmec (SCAL only)
    for (int r = 0; r < NSUM; ++r) { S[r] = 0.0; T[r] = 0.0; }
    if constexpr (SCAL)
        for (int r = 0; r < NSUM; ++r) P[r] = 0.0;
    for (int q = 0; q < mn; ++q) {
        const double m = p.xm[q], n = p.xn[q];
        double sa, ca;
        sincos(m * th - n * phi, &sa, &ca);
        const double r = tm[q], z = tm[mn + q], l = tm[2 * mn + q], rs = tm[3 * mn + q], zs = tm[4 * mn + q], ls = tm[5 * mn + q];
        S[S_R] += r * ca;        T[S_R] -= r * m * sa;
        S[S_Rs] += rs * ca;      T[S_Rs] -= rs * m * sa;
        S[S_Rt] -= r * m * sa;   T[S_Rt] -= r * m * m * ca;
        S[S_Rp] += r * n * sa;   T[S_Rp] += r * n * m * ca;
        S[S_Zs] += zs * sa;      T[S_Zs] += zs * m * ca;
        S[S_Zt] += z * m * ca;   T[S_Zt] -= z * m * m * sa;
        S[S_Zp] -= z * n * ca;   T[S_Zp] += z * n * m * sa;
        S[S_Ls] += ls * sa;      T[S_Ls] += ls * m * ca;
        S[S_Lt] += l * m * ca;   T[S_Lt] -= l * m * m * sa;
        S[S_Lp] -= l * n * ca;   T[S_Lp] += l * n * m * sa;
        if constexpr (SCAL) {
            P[S_R] += r * n * sa;    P[S_Rs] += rs * n * sa;  P[S_Rt] += r * m * n * ca;  P[S_Rp] -= r * n * n * ca;
            P[S_Zs] -= zs * n * ca;  P[S_Zt] += z * m * n * sa;  P[S_Zp] -= z * n * n * sa;
            P[S_Ls] -= ls * n * ca;  P[S_Lt] += l * m * n * sa;  P[S_Lp] -= l * n * n * sa;
        }
    }
    for (int q = 0; q < mq; ++q) {
        const double m = p.xm_nyq[q], n = p.xn_nyq[q];
        double sa, ca;
        sincos(m * th - n * phi, &sa, &ca);
        const double g = tq[q], b = tq[mq + q], bs = tq[2 * mq + q], bv = tq[3 * mq + q], s_ = tq[4 * mq + q], u_ = tq[5 * mq + q], v_ = tq[6 * mq + q];
        S[S_sqrtg] += g * ca;    T[S_sqrtg] -= g * m * sa;
        S[S_B] += b * ca;        T[S_B] -= b * m * sa;
        S[S_Bs] += bs * ca;      T[S_Bs] -= bs * m * sa;
        S[S_Bt] -= b * m * sa;   T[S_Bt] -= b * m * m * ca;
        S[S_Bp] += b * n * sa;   T[S_Bp] += b * n * m * ca;
        S[S_Bsupp] += bv * ca;   T[S_Bsupp] -= bv * m * sa;
        S[S_Bsubs] += s_ * sa;   T[S_Bsubs] += s_ * m * ca;
        S[S_Bsubt] += u_ * ca;   T[S_Bsubt] -= u_ * m * sa;
        S[S_Bsubp] += v_ * ca;   T[S_Bsubp] -= v_ * m * sa;
        if constexpr (SCAL) {
            P[S_sqrtg] += g * n * sa;  P[S_B] += b * n * sa;  P[S_Bs] += bs * n * sa;  P[S_Bt] += b * m * n * ca;
            P[S_Bp] -= b * n * n * ca;  P[S_Bsupp] += bv * n * sa;  P[S_Bsubs] -= s_ * n * ca;  P[S_Bsubt] += u_ * n * sa;
            P[S_Bsubp] += v_ * n * sa;
        }
    }
    if constexpr (!SCAL) {
        // v_r = d Phi / d S_r by 19 forward sweeps; dPhi/dtheta_vmec = sum_r v_r T_r
        double* w = p.work + (size_t)js * (NSUM + 3) * p.nl + jl;
        double dth = 0.0;
        for (int r = 0; r < NSUM; ++r) {
            D1 Sd[NSUM];
            for (int q = 0; q < NSUM; ++q) Sd[q] = D1(S[q], q == r ? 1.0 : 0.0);
            const double v = phi_point(Sd, k).d;
            w[(size_t)r * p.nl] = v;
            dth = fma(v, T[r], dth);
        }
        w[(size_t)NSUM * p.nl] = -dth / (1.0 + S[S_Lt]);          // weight of d(lmns) sin a (implicit theta_vmec)
        w[(size_t)(NSUM + 1) * p.nl] = th;
        w[(size_t)(NSUM + 2) * p.nl] = phi;
    } else {
        // total d Phi_j / dx, one sweep per scalar x; only iota moves the point (phi, hence sin / cos phi and the sums)
        const double dphi_di = -k.dphi / k.iota;
        const double th_phi = -S[S_Lp] / (1.0 + S[S_Lt]);
        double* ws = p.work_scal + (size_t)js * NSX * p.nl + jl;
        for (int x = 0; x < NSX; ++x) {
            const auto seed = [x](int which, double d) { return x == which ? d : 0.0; };
            const double e = seed(1, dphi_di);
            PointConst<D1> kd;
            kd.sp = D1(k.sp, k.cp * e); kd.cp = D1(k.cp, -k.sp * e); kd.dphi = D1(k.dphi, e);
            kd.s_val = D1(k.s_val, seed(0, 1.0)); kd.iota = D1(k.iota, seed(1, 1.0)); kd.d_iota = D1(k.d_iota, seed(2, 1.0));
            kd.dpds = D1(k.dpds, seed(3, 1.0)); kd.shat = D1(k.shat, seed(4, 1.0));
            kd.psi_e = D1(k.psi_e, seed(5, -1.0 / (2.0 * 3.141592653589793)));         // psi_e = -phiedge / 2 pi
            kd.L_ref = D1(k.L_ref, seed(6, 1.0));                                      // L_ref = Aminor_p
            kd.th0 = k.th0; kd.dP = k.dP; kd.sg = k.sg; kd.sc = k.sc; kd.sf = k.sf; kd.qw = k.qw;
            D1 Sd[NSUM];
            for (int r = 0; r < NSUM; ++r) Sd[r] = D1(S[r], (P[r] + T[r] * th_phi) * e);
            ws[(size_t)x * p.nl] = phi_point(Sd, kd).d;
        }
    }
}

// stage B: one thread per (surface, mode); modes 0 .. mnmax-1 of the (R, Z, lambda) set, then the Nyquist set
__global__ void __launch_bounds__(128)
geo_adjoint_mode_kernel(const GeoAdjParams p) {
    const int js = blockIdx.y;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int mn = p.mnmax, mq = p.mnmax_nyq;
    if (q >= mn + mq) return;
    const bool nyq = q >= mn;
    const int kq = nyq ? q - mn : q;
    const double m = nyq ? p.xm_nyq[kq] : p.xm[kq], n = nyq ? p.xn_nyq[kq] : p.xn[kq];
    const double* w = p.work + (size_t)js * (NSUM + 3) * p.nl;
    const double* th = w + (size_t)(NSUM + 1) * p.nl;
    const double* ph = w + (size_t)(NSUM + 2) * p.nl;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0, a4 = 0, a5 = 0, a6 = 0;
    for (int j = 0; j < p.nl; ++j) {
        double sa, ca;
        sincos(m * th[j] - n * ph[j], &sa, &ca);
#define V(r) w[(size_t)(r) * p.nl + j]
        if (!nyq) {
            a0 += V(S_R) * ca - m * V(S_Rt) * sa + n * V(S_Rp) * sa;                 // rmnc
            a1 += m * V(S_Zt) * ca - n * V(S_Zp) * ca;                                // zmns
            a2 += m * V(S_Lt) * ca - n * V(S_Lp) * ca + V(NSUM) * sa;                 // lmns (explicit + through theta_vmec)
            a3 += V(S_Rs) * ca;                                                       // d_rmnc_d_s
            a4 += V(S_Zs) * sa;                                                       // d_zmns_d_s
            a5 += V(S_Ls) * sa;                                                       // d_lmns_d_s
        } else {
            a0 += V(S_sqrtg) * ca;                                                    // gmnc
            a1 += V(S_B) * ca - m * V(S_Bt) * sa + n * V(S_Bp) * sa;                  // bmnc
            a2 += V(S_Bs) * ca;                                                       // d_bmnc_d_s
            a3 += V(S_Bsupp) * ca;                                                    // bsupvmnc
            a4 += V(S_Bsubs) * sa;                                                    // bsubsmns
            a5 += V(S_Bsubt) * ca;                                                    // bsubumnc
            a6 += V(S_Bsubp) * ca;                                                    // bsubvmnc
        }
#undef V
    }
    if (!nyq) {
        double* g = p.grad_mn + (size_t)js * IBS_TAB_MN_ROWS * mn + kq;
        g[0] = a0; g[mn] = a1; g[2 * mn] = a2; g[3 * mn] = a3; g[4 * mn] = a4; g[5 * mn] = a5;
    } else {
        double* g = p.grad_nyq + (size_t)js * IBS_TAB_NYQ_ROWS * mq + kq;
        g[0] = a0; g[mq] = a1; g[2 * mq] = a2; g[3 * mq] = a3; g[4 * mq] = a4; g[5 * mq] = a5; g[6 * mq] = a6;
    }
}

// stage B of the scalar sweeps: one thread per (surface, scalar), the sum over the line in point order
__global__ void __launch_bounds__(128)
geo_adjoint_scal_sum_kernel(const GeoAdjParams p) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.ns * NSX) return;
    const int js = t / NSX, x = t - js * NSX;
    const double* ws = p.work_scal + (size_t)t * p.nl;
    double a = 0.0;
    for (int j = 0; j < p.nl; ++j) a += ws[j];
    if (x < 5) p.grad_scal[(size_t)js * IBS_NSCAL + x] = a;
    else p.grad_glob[(size_t)js * 2 + (x - 5)] = a;
    if (x == 0)                                                    // pressure and the spare columns: K1 does not read them
        for (int c = 5; c < IBS_NSCAL; ++c) p.grad_scal[(size_t)js * IBS_NSCAL + c] = 0.0;
}

int geometry_adjoint_dispatch(const double* tab_mn, const double* tab_nyq, const double* scal, const double* xm, const double* xn,
                              const double* xm_nyq, const double* xn_nyq, int ns, int mnmax, int mnmax_nyq, double phiedge,
                              double aminor_p, const double* alpha, const double* theta, int nl, double phi_center,
                              const double* theta0, const double* dPdrho, const double* sg, const double* sc, const double* sf,
                              const double* Q, double* grad_mn, double* grad_nyq, double* grad_scal, double* grad_glob,
                              cudaStream_t st) {
    if (ns == 0) return IBS_OK;
    const bool scal_out = grad_scal != nullptr;
    GeoAdjParams p;
    p.tab_mn = tab_mn; p.tab_nyq = tab_nyq; p.scal = scal; p.xm = xm; p.xn = xn; p.xm_nyq = xm_nyq; p.xn_nyq = xn_nyq;
    p.ns = ns; p.mnmax = mnmax; p.mnmax_nyq = mnmax_nyq; p.nl = nl; p.alpha = alpha; p.theta = theta; p.theta0 = theta0; p.dPdrho = dPdrho;
    p.sg = sg; p.sc = sc; p.sf = sf; p.Q = Q; p.phi_center = phi_center; p.psi_e = -phiedge / (2.0 * 3.141592653589793); p.L_ref = aminor_p;
    p.grad_mn = grad_mn; p.grad_nyq = grad_nyq; p.grad_scal = grad_scal; p.grad_glob = grad_glob;
    keep_pool_cached();
    const size_t nwork = (size_t)ns * (NSUM + 3) * nl;
    IBS_CUDA_CHECK(cudaMallocAsync((void**)&p.work, (nwork + (scal_out ? (size_t)ns * NSX * nl : 0)) * sizeof(double), st));
    p.work_scal = scal_out ? p.work + nwork : nullptr;
    const long long npt = (long long)ns * nl;
    const unsigned npb = (unsigned)((npt + 127) / 128);
    geo_adjoint_point_kernel<false><<<npb, 128, 0, st>>>(p);
    if (scal_out) geo_adjoint_point_kernel<true><<<npb, 128, 0, st>>>(p);
    int rc = (cudaGetLastError() == cudaSuccess) ? IBS_OK : IBS_ERR_CUDA;
    if (rc == IBS_OK) {
        geo_adjoint_mode_kernel<<<dim3((mnmax + mnmax_nyq + 127) / 128, ns), 128, 0, st>>>(p);
        if (scal_out) geo_adjoint_scal_sum_kernel<<<(ns * NSX + 127) / 128, 128, 0, st>>>(p);
        if (cudaGetLastError() != cudaSuccess) rc = IBS_ERR_CUDA;
    }
    if (rc != IBS_OK) set_error("geometry adjoint kernel launch failed");
    cudaFreeAsync(p.work, st);
    return rc;
}

}  // namespace ibs
