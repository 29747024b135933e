// Forward-mode algebra of K1's pointwise epilogue, shared by the reverse-mode geometry (ibs_geometry_adjoint.cu) and the
// alpha-tangent of K1 (ibs_geometry.cu, geometry_tangent_kernel).
#pragma once
#include "ibs_common.cuh"

namespace ibs {

// ---- forward-mode scalar: value + one directional derivative -----------------------------------------------------------
struct D1 {
    double v, d;
    __device__ __forceinline__ D1() : v(0.0), d(0.0) {}
    __device__ __forceinline__ D1(double v_) : v(v_), d(0.0) {}
    __device__ __forceinline__ D1(double v_, double d_) : v(v_), d(d_) {}
};
__device__ __forceinline__ D1 operator+(D1 a, D1 b) { return {a.v + b.v, a.d + b.d}; }
__device__ __forceinline__ D1 operator-(D1 a, D1 b) { return {a.v - b.v, a.d - b.d}; }
__device__ __forceinline__ D1 operator-(D1 a) { return {-a.v, -a.d}; }
__device__ __forceinline__ D1 operator*(D1 a, D1 b) { return {a.v * b.v, a.d * b.v + a.v * b.d}; }
__device__ __forceinline__ D1 operator/(D1 a, D1 b) { const double q = a.v / b.v; return {q, (a.d - q * b.d) / b.v}; }
__device__ __forceinline__ D1 dabs(D1 a) { return a.v < 0.0 ? D1{-a.v, -a.d} : a; }
// the per-surface constants are double (table sweeps) or D1 (scalar sweeps)
__device__ __forceinline__ double cabs(double a) { return fabs(a); }
__device__ __forceinline__ D1 cabs(D1 a) { return dabs(a); }
__device__ __forceinline__ double csqrt(double a) { return sqrt(a); }
__device__ __forceinline__ D1 csqrt(D1 a) { const double r = sqrt(a.v); return {r, 0.5 * a.d / r}; }
__device__ __forceinline__ double cval(double a) { return a; }
__device__ __forceinline__ double cval(D1 a) { return a.v; }

// the 19 mode sums of one point (utils.py:432-468)
constexpr int NSUM = 19;
enum { S_R, S_Rs, S_Rt, S_Rp, S_Zs, S_Zt, S_Zp, S_Ls, S_Lt, S_Lp, S_sqrtg, S_B, S_Bs, S_Bt, S_Bp, S_Bsupp, S_Bsubs, S_Bsubt, S_Bsubp };

template <class C>
struct PointConst {
    C sp, cp, dphi;                       // sin / cos(phi), phi - phi_center
    C iota, d_iota, dpds, shat, s_val, psi_e, L_ref;
    double th0, dP, sg, sc, sf, qw;       // theta0, dPdrho, the three sensitivities of this point, Q / (2 N) (reverse mode only)
};

// The eight base arrays of one point (IBS_BASE_* order) as functions of the 19 mode sums: the pointwise algebra of
// geo_point_epilogue (ibs_geometry.cu) on D1
template <class C>
__device__ __forceinline__ void base_point(const D1 (&S)[NSUM], const PointConst<C>& k, D1 (&out)[IBS_NBASE]) {
    const D1 R = S[S_R], R_s = S[S_Rs], R_t = S[S_Rt], R_p = S[S_Rp], Z_s = S[S_Zs], Z_t = S[S_Zt], Z_p = S[S_Zp];
    const D1 L_s = S[S_Ls], L_t = S[S_Lt], L_p = S[S_Lp];
    const D1 sqrtg = S[S_sqrtg], B = S[S_B], B_s = S[S_Bs], B_t = S[S_Bt], B_p = S[S_Bp], Bsup_p = S[S_Bsupp];
    const D1 Bsub_s = S[S_Bsubs], Bsub_t = S[S_Bsubt], Bsub_p = S[S_Bsubp];
    const D1 sp = k.sp, cp = k.cp;
    const D1 X_t = R_t * cp, X_p = R_p * cp - R * sp, X_s = R_s * cp;
    const D1 Y_t = R_t * sp, Y_p = R_p * sp + R * cp, Y_s = R_s * sp;
    const D1 isg = D1(1.0) / sqrtg;
    const D1 gsx = (Y_t * Z_p - Z_t * Y_p) * isg, gsy = (Z_t * X_p - X_t * Z_p) * isg, gsz = (X_t * Y_p - Y_t * X_p) * isg;
    const D1 gtx = (Y_p * Z_s - Z_p * Y_s) * isg, gty = (Z_p * X_s - X_p * Z_s) * isg, gtz = (X_p * Y_s - Y_p * X_s) * isg;
    const D1 gpx = (Y_s * Z_t - Z_s * Y_t) * isg, gpy = (Z_s * X_t - X_s * Z_t) * isg, gpz = (X_s * Y_t - Y_s * X_t) * isg;
    const D1 psi_e = k.psi_e;
    const D1 a_s = L_s - D1(k.dphi * k.d_iota);
    const D1 a_t = D1(1.0) + L_t, a_p = L_p - D1(k.iota);
    const D1 gax = a_s * gsx + (a_t * gtx + a_p * gpx), gay = a_s * gsy + (a_t * gty + a_p * gpy), gaz = a_s * gsz + (a_t * gtz + a_p * gpz);
    const D1 gqx = gsx * psi_e, gqy = gsy * psi_e, gqz = gsz * psi_e;
    const D1 lpi = a_p;
    const D1 BxgB_ga = (Bsub_s * B_t * lpi + Bsub_t * B_p * a_s + Bsub_p * B_s * a_t - Bsub_p * B_t * a_s - Bsub_t * B_s * lpi -
                        Bsub_s * B_p * a_t) * isg;
    const D1 ga_ga = gax * gax + gay * gay + gaz * gaz, ga_gq = gax * gqx + gay * gqy + gaz * gqz, gq_gq = gqx * gqx + gqy * gqy + gqz * gqz;
    const D1 BxgB_gq = (Bsub_t * B_p - Bsub_p * B_t) * isg * psi_e;
    const C L_ref = k.L_ref, B_ref = 2.0 * cabs(k.psi_e) / (L_ref * L_ref);
    const double sgn = (cval(k.psi_e) > 0.0) ? 1.0 : ((cval(k.psi_e) < 0.0) ? -1.0 : 0.0);
    const C sqrt_s = csqrt(k.s_val);
    const double mu0 = 4.0 * 3.141592653589793 * 1.0e-7;
    const D1 B3 = B * B * B;
    out[IBS_BASE_BMAG] = B / D1(B_ref);
    out[IBS_BASE_GRADPAR] = D1(L_ref * k.iota) * Bsup_p / B;
    out[IBS_BASE_GDS2] = ga_ga * D1(L_ref * L_ref * k.s_val);
    out[IBS_BASE_GDS21] = ga_gq * D1(k.shat / B_ref);
    out[IBS_BASE_GDS22] = gq_gq * D1(k.shat * k.shat / (L_ref * L_ref * B_ref * B_ref * k.s_val));
    const D1 gbdrift = D1(-2.0 * B_ref * L_ref * L_ref * sqrt_s * sgn) * BxgB_ga / B3;
    out[IBS_BASE_GBDRIFT] = gbdrift;
    out[IBS_BASE_CVDRIFT0] = D1(-2.0 * k.shat * sgn / sqrt_s) * BxgB_gq / B3;         // cvdrift0 = gbdrift0 (utils.py:720)
    out[IBS_BASE_CVDRIFT] = gbdrift - D1(2.0 * B_ref * L_ref * L_ref * sqrt_s * mu0 * k.dpds * sgn / k.psi_e) / (B * B);
}

}  // namespace ibs
