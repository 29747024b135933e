// K1: field-line geometry assembly.  Replaces the hot-path subset of vmec_fieldlines
// (/root/reference/utils.py:161-864): theta_vmec root solve (:391-416), the 19 Fourier mode sums the
// ballooning path needs (:420-468), the Cartesian dual basis and drifts (:474-658) and the GS2
// normalisations (:662-720).  fp64 throughout; FP64-pipe bound (no tensor cores: the contraction has
// only 10 / 9 output rows per mode set, a poor DMMA shape, and the trig generation is not a GEMM).
//
// Layout / mapping
//   * One CTA works on one surface at a time; the surface's Fourier tables are re-packed on the fly
//     (pack kernels below) into a dense (m, n) grid  tab[m][n_idx][ROW]  so that the inner n loop can be
//     fully unrolled with compile-time signs and n-weights, and are staged into shared memory with one
//     TMA bulk copy (cp.async.bulk + mbarrier) per table.  All threads then read the same coefficient
//     at the same time: broadcast LDS.128, no bank conflicts.
//   * One thread = one point of a field line.  cos/sin(n nfp phi) for n = 0..NT live in registers
//     (angle-addition recurrence from one sincos), cos/sin(m theta) advance by recurrence in the m loop,
//     so cos(m theta - n phi) costs 2 FMA-pairs instead of a sincos per mode: 30 sincos per point
//     instead of 634 for NCSX.
//   * The Newton solve for theta_vmec uses the n-sums A_m = sum_n l_mn cos(n phi), B_m = sum_n l_mn
//     sin(n phi), which are fixed along the iteration, so each iteration costs O(mpol), not O(mnmax).
#include <mutex>
#include <vector>
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "ibs_common.cuh"
#include "ibs_geometry_ad.cuh"

namespace ibs {

constexpr int GEO_THREADS = 128;          // axisymmetric tables: 128-point tiles
// Round 1's one-point-per-thread 3-D instantiations (kept for comparison, IBS_GEO3D=0).  Measured in round 2: 512-thread
// CTAs at 128 registers (16 warps / SM) and A_m, B_m in shared memory are 3-9 % SLOWER (NCSX 2.94 -> 3.23 ms, HBERG 92 -> 101 ms):
// the kernel is bound by the shared-memory data pipe (0.86 wavefronts / clk / SM), not by latency -- see geometry3d_kernel.
#ifndef IBS_GEO_THREADS_3D
#define IBS_GEO_THREADS_3D 128
#endif
#ifndef IBS_GEO_FAST_EPILOGUE
#define IBS_GEO_FAST_EPILOGUE 0      // see geo_point_epilogue: K1 -2 %, but the solver then ran 8-10 % SLOWER on the (2-3 ulp different) arrays -- left off
#endif
#ifndef IBS_GEO_KC_INLOOP
#define IBS_GEO_KC_INLOOP 0
#endif
#ifndef IBS_GEO_MINB
#define IBS_GEO_MINB 1
#endif
#ifndef IBS_GEO_NROWS_DERIVED
#define IBS_GEO_NROWS_DERIVED 1
#endif
#ifndef IBS_GEO_SMEM_NEWTON
#define IBS_GEO_SMEM_NEWTON 0
#endif
constexpr int GEO_THREADS_3D = IBS_GEO_THREADS_3D;
constexpr int GEO_SMEM_NEWTON_MAX_M = 16;  // A_m, B_m live in shared memory when mpol + 1 <= this (2 * 16 * 512 * 8 B = 128 KB), else in local memory
template <int NT1> struct GeoThreads { static constexpr int value = (NT1 > 0) ? GEO_THREADS_3D : GEO_THREADS; };
constexpr int ROW_MN = 10;    // r, n r, r_s, z, n z, z_s, l, n l, l_s, (pad)
constexpr int ROW_NYQ = 8;    // g, b, n b, b_s, bsupv, bsubs, bsubu, bsubv
// 3-D equilibria use a paired layout [m][|n|][row][E, O] (E = v(+n) + v(-n), O = v(+n) - v(-n)): with
//   sum_n v_n cos(m th - n ph) = cos(m th) A + sin(m th) B,   sum_n v_n sin(m th - n ph) = sin(m th) A - cos(m th) B,
//   A = v_0 + sum_{k>0} E_k cos(k nfp ph),  B = sum_{k>0} O_k sin(k nfp ph),
// a mode costs one FMA per table row (no per-mode angle update): ~30 % fewer FP64 instructions than the dense +-n grid.
constexpr int ROWP_MN = 18, ROWP_NYQ = 16;
constexpr int MAX_M_NEWTON = 96;

struct GeoParams {
    const double* pk_mn;    // [ns][M1][W1][ROW_MN]
    const double* pk_nyq;   // [ns][M2][W2][ROW_NYQ]
    const double* scal;     // [ns][8]
    const double* alpha; int nalpha; int alpha_per_surface;
    const double* theta; int nl;
    int ns, M1, M2;         // number of m values in each set
    int nfp;                // toroidal stride of the packed n index
    double phi_center, psi_e, L_ref;
    double* base_out; double* theta_vmec_out; int* info_out;
    int fold;               // axisymmetric tables: allow the periodicity fold (IBS_GEO_FOLD=0 turns it off)
};

// ---- pack kernels: (ns, rows, mn) tables -> dense (m, n_idx) grid with the n-weights folded in -----------
__global__ void pack_mn_kernel(const double* __restrict__ tab, const int* __restrict__ mode_m, const int* __restrict__ mode_n,
                               int ns, int mnmax, int M1, int W1, int NT1, int nfp, double* __restrict__ out) {
    const int s = blockIdx.x;                                   // surfaces on x (up to 2^31 - 1 of them)
    const int k = blockIdx.y * blockDim.x + threadIdx.x;
    if (k >= mnmax) return;
    const int m = mode_m[k], nn = mode_n[k];          // nn = n / nfp
    const double* t = tab + (size_t)s * 6 * mnmax;
    const double n = (double)(nn * nfp);
    const double r = t[0 * mnmax + k], z = t[1 * mnmax + k], l = t[2 * mnmax + k];
    const double v[9] = {r, n * r, t[3 * mnmax + k], z, n * z, t[4 * mnmax + k], l, n * l, t[5 * mnmax + k]};
    // duplicates in the mode list are legal (they add up)
    if (NT1 == 0) {
        double* o = out + (((size_t)s * M1 + m) * W1 + (nn + NT1)) * ROW_MN;
        for (int j = 0; j < 9; ++j) atomicAdd(o + j, v[j]);
    } else {
        // paired layout [m][|n|][row][E, O]:  E = v(+n) + v(-n),  O = v(+n) - v(-n)
        const int ak = nn < 0 ? -nn : nn;
        const double sg = nn > 0 ? 1.0 : (nn < 0 ? -1.0 : 0.0);
        double* o = out + (((size_t)s * M1 + m) * (NT1 + 1) + ak) * ROWP_MN;
        for (int j = 0; j < 9; ++j) { atomicAdd(o + 2 * j, v[j]); atomicAdd(o + 2 * j + 1, sg * v[j]); }
    }
}
__global__ void pack_nyq_kernel(const double* __restrict__ tab, const int* __restrict__ mode_m, const int* __restrict__ mode_n,
                                int ns, int mnmax, int M2, int W2, int NT2, int nfp, double* __restrict__ out) {
    const int s = blockIdx.x;                                   // surfaces on x (up to 2^31 - 1 of them)
    const int k = blockIdx.y * blockDim.x + threadIdx.x;
    if (k >= mnmax) return;
    const int m = mode_m[k], nn = mode_n[k];
    const double* t = tab + (size_t)s * 7 * mnmax;
    const double n = (double)(nn * nfp);
    const double b = t[1 * mnmax + k];
    const double v[8] = {t[0 * mnmax + k], b, n * b, t[2 * mnmax + k], t[3 * mnmax + k], t[4 * mnmax + k], t[5 * mnmax + k], t[6 * mnmax + k]};
    if (NT2 == 0) {
        double* o = out + (((size_t)s * M2 + m) * W2 + (nn + NT2)) * ROW_NYQ;
        for (int j = 0; j < 8; ++j) atomicAdd(o + j, v[j]);
    } else {
        const int ak = nn < 0 ? -nn : nn;
        const double sg = nn > 0 ? 1.0 : (nn < 0 ? -1.0 : 0.0);
        double* o = out + (((size_t)s * M2 + m) * (NT2 + 1) + ak) * ROWP_NYQ;
        for (int j = 0; j < 8; ++j) { atomicAdd(o + 2 * j, v[j]); atomicAdd(o + 2 * j + 1, sg * v[j]); }
    }
}

// cos/sin(m theta - n phi) for one n_idx with compile-time sign
template <int SGN> __device__ __forceinline__ void angle(double cm, double sm, double cn, double sn, double& ca, double& sa) {
    if (SGN >= 0) { ca = fma(cm, cn, sm * sn); sa = fma(sm, cn, -(cm * sn)); }      // n >= 0: m th - |n| ph
    else          { ca = fma(cm, cn, -(sm * sn)); sa = fma(sm, cn, cm * sn); }      // n <  0: m th + |n| ph
}

// The 19 mode sums of one point (utils.py:432-468) handed to the pointwise epilogue
struct GeoSums {
    double R, R_s, R_t, R_p, Z_s, Z_t, Z_p, L_s, L_t, L_p;
    double sqrtg, B, B_s, B_t, B_p, Bsup_p, Bsub_s, Bsub_t, Bsub_p;
};

// Pointwise algebra of one point (dual basis, grad alpha / psi, drifts, GS2 normalisations: utils.py:474-720) and the
// stores of its eight base-array entries
__device__ __forceinline__ void geo_point_epilogue(const GeoParams& p, const GeoSums& gs_, int js, int ja, int jl, double phi, double th,
                                                   int nit, bool ok, double s_val, double iota, double d_iota, double dpds, double shat) {
    const double R = gs_.R, R_s = gs_.R_s, R_t = gs_.R_t, R_p = gs_.R_p, Z_s = gs_.Z_s, Z_t = gs_.Z_t, Z_p = gs_.Z_p;
    const double L_s = gs_.L_s, L_t = gs_.L_t, L_p = gs_.L_p;
    const double sqrtg = gs_.sqrtg, B = gs_.B, B_s = gs_.B_s, B_t = gs_.B_t, B_p = gs_.B_p, Bsup_p = gs_.Bsup_p;
    const double Bsub_s = gs_.Bsub_s, Bsub_t = gs_.Bsub_t, Bsub_p = gs_.Bsub_p;
    // ---- Cartesian dual basis (utils.py:480-508)
    double sp, cp;
    sincos(phi, &sp, &cp);
    const double X_t = R_t * cp, X_p = R_p * cp - R * sp, X_s = R_s * cp;
    const double Y_t = R_t * sp, Y_p = R_p * sp + R * cp, Y_s = R_s * sp;
    const double isg = 1.0 / sqrtg;
    const double gsx = (Y_t * Z_p - Z_t * Y_p) * isg, gsy = (Z_t * X_p - X_t * Z_p) * isg, gsz = (X_t * Y_p - Y_t * X_p) * isg;
    const double gtx = (Y_p * Z_s - Z_p * Y_s) * isg, gty = (Z_p * X_s - X_p * Z_s) * isg, gtz = (X_p * Y_s - Y_p * X_s) * isg;
    const double gpx = (Y_s * Z_t - Z_s * Y_t) * isg, gpy = (Z_s * X_t - X_s * Z_t) * isg, gpz = (X_s * Y_t - Y_s * X_t) * isg;
    // grad psi, grad alpha (utils.py:515-538)
    const double psi_e = p.psi_e;
    const double a_s = L_s - (phi - p.phi_center) * d_iota;
    const double a_t = 1.0 + L_t, a_p = -iota + L_p;
    const double gax = a_s * gsx + (a_t * gtx + a_p * gpx);
    const double gay = a_s * gsy + (a_t * gty + a_p * gpy);
    const double gaz = a_s * gsz + (a_t * gtz + a_p * gpz);
    const double gqx = gsx * psi_e, gqy = gsy * psi_e, gqz = gsz * psi_e;
    // drifts (utils.py:603-618, 646-650)
    const double lpi = L_p - iota;
    const double BxgB_ga = (Bsub_s * B_t * lpi + Bsub_t * B_p * a_s + Bsub_p * B_s * a_t - Bsub_p * B_t * a_s -
                            Bsub_t * B_s * lpi - Bsub_s * B_p * a_t) * isg;
    const double ga_ga = gax * gax + gay * gay + gaz * gaz;
    const double ga_gq = gax * gqx + gay * gqy + gaz * gqz;
    const double gq_gq = gqx * gqx + gqy * gqy + gqz * gqz;
    const double BxgB_gq = (Bsub_t * B_p - Bsub_p * B_t) * isg * psi_e;
    // GS2 normalisations (utils.py:662-720)
    const double L_ref = p.L_ref, B_ref = 2.0 * fabs(psi_e) / (L_ref * L_ref);
    const double sgn = (psi_e > 0.0) ? 1.0 : ((psi_e < 0.0) ? -1.0 : 0.0);
    const double sqrt_s = sqrt(s_val);
    const double mu0 = 4.0 * 3.141592653589793 * 1.0e-7;
#if IBS_GEO_FAST_EPILOGUE
    // Same formulas with ONE point-dependent reciprocal (1 / B) instead of four divisions by B, B^3, B^3 sqrt(s), psi B^2; the other
    // divisors are per-surface constants (their reciprocals leave the fold loop).  2-3 ulp instead of 1 on these entries -- the
    // epilogue runs 4-5 times per Newton solve on folded axisymmetric grids, where it was a third of the kernel.
    // MEASURED (D3D bench): K1 0.588 -> 0.577 ms, but scan2_solve_kernel on the resulting arrays 2.67 -> 2.93 ms with the SAME
    // executed instructions (1.6013e9 vs 1.6020e9), the same stalls per issue and the same warps active (ncu): not understood;
    // the IEEE-division form stays the default.
    const double iB = 1.0 / B, iB2 = iB * iB, iB3 = iB2 * iB;
    const double iBref = 1.0 / B_ref, isqs = 1.0 / sqrt_s;
    const double bmag = B * iBref;
    const double gradpar = L_ref * (iota * Bsup_p) * iB;
    const double gds2 = ga_ga * L_ref * L_ref * s_val;
    const double gds21 = ga_gq * shat * iBref;
    const double gds22 = gq_gq * (shat * shat / (L_ref * L_ref * B_ref * B_ref * s_val));
    const double gbdrift = (-2.0 * B_ref * L_ref * L_ref * sqrt_s * sgn) * BxgB_ga * iB3;
    const double gbdrift0 = (-2.0 * shat * isqs * sgn) * BxgB_gq * iB3;
    const double cvdrift = gbdrift - (2.0 * B_ref * L_ref * L_ref * sqrt_s * mu0 * dpds * sgn / psi_e) * iB2;
#else
    const double B3 = B * B * B;
    const double bmag = B / B_ref;
    const double gradpar = L_ref * (iota * Bsup_p) / B;
    const double gds2 = ga_ga * L_ref * L_ref * s_val;
    const double gds21 = ga_gq * shat / B_ref;
    const double gds22 = gq_gq * shat * shat / (L_ref * L_ref * B_ref * B_ref * s_val);
    const double gbdrift = -1.0 * 2.0 * B_ref * L_ref * L_ref * sqrt_s * BxgB_ga / B3 * sgn;
    const double gbdrift0 = -1.0 * BxgB_gq * 2.0 * shat / (B3 * sqrt_s) * sgn;
    const double cvdrift = gbdrift - 2.0 * B_ref * L_ref * L_ref * sqrt_s * mu0 * dpds * sgn / (psi_e * B * B);
#endif

    const size_t line = (size_t)js * p.nalpha + ja;
    double* o = p.base_out + line * IBS_NBASE * p.nl + jl;
    o[(size_t)IBS_BASE_BMAG * p.nl] = bmag;
    o[(size_t)IBS_BASE_GRADPAR * p.nl] = gradpar;
    o[(size_t)IBS_BASE_CVDRIFT * p.nl] = cvdrift;
    o[(size_t)IBS_BASE_CVDRIFT0 * p.nl] = gbdrift0;      // cvdrift0 = gbdrift0 (utils.py:720)
    o[(size_t)IBS_BASE_GDS2 * p.nl] = gds2;
    o[(size_t)IBS_BASE_GDS21 * p.nl] = gds21;
    o[(size_t)IBS_BASE_GDS22 * p.nl] = gds22;
    o[(size_t)IBS_BASE_GBDRIFT * p.nl] = gbdrift;
    if (p.theta_vmec_out) p.theta_vmec_out[line * p.nl + jl] = th;
    if (p.info_out) atomicMax(p.info_out + line, nit | (ok ? 0 : (1 << 16)));
}

template <int NT1, int NT2>
#if IBS_GEO_MINB > 1
__global__ void __launch_bounds__(GeoThreads<NT1>::value, (NT1 > 0) ? IBS_GEO_MINB : 1)
#else
__global__ void __launch_bounds__(GeoThreads<NT1>::value)          // (a min-blocks argument of 1 lets ptxas take 254 registers: 3 instead of 4 CTAs / SM on the axisymmetric path)
#endif
geometry_kernel(const GeoParams p) {
    constexpr int W1 = 2 * NT1 + 1, W2 = 2 * NT2 + 1, NT = (NT1 > NT2 ? NT1 : NT2);
    constexpr int GEO_THREADS = GeoThreads<NT1>::value;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    double* s_mn = reinterpret_cast<double*>(smem_raw + 16);
    const int n_mn = (NT1 > 0) ? p.M1 * (NT1 + 1) * ROWP_MN : p.M1 * W1 * ROW_MN;
    const int n_nyq = (NT2 > 0) ? p.M2 * (NT2 + 1) * ROWP_NYQ : p.M2 * W2 * ROW_NYQ;
    double* s_nyq = s_mn + n_mn;
    const int tid = threadIdx.x;
    // Periodicity fold (axisymmetric tables only).  Every mode sum is 2 pi-periodic in theta_vmec and does not depend on phi,
    // and theta_vmec(theta_pest + 2 pi) = theta_vmec(theta_pest) + 2 pi, so grid points one poloidal turn apart share their
    // Newton solve and their 19 sums; only the pointwise epilogue (secular shear term, phi) is per point.  The reference's
    // own grids are commensurate: theta = linspace(-f pi, f pi, 2 mpol f + 1) (ball_scan.py:204-208) has 2 mpol points per
    // turn.  Checked on the data, not assumed: P = rint(2 pi / (theta[1] - theta[0])) is used only if EVERY point satisfies
    // theta[j] = theta[j mod P] + 2 pi (j div P) to 2e-12 (the grid need not be uniform).
    int P = p.nl;
    if constexpr (NT1 == 0 && NT2 == 0) {
        if (p.fold && p.nl >= 3) {
            const double TWO_PI = 6.283185307179586;
            const double h0 = p.theta[1] - p.theta[0];
            const double pf = (h0 > 0.0) ? TWO_PI / h0 : 0.0;
            const int Pc = (pf >= 2.0 && pf < (double)p.nl) ? (int)rint(pf) : 0;
            bool okf = Pc >= 2 && Pc < p.nl;
            if (okf)
                for (int j = tid; j < p.nl; j += GEO_THREADS) {
                    const int q = j / Pc, r = j - q * Pc;
                    okf &= fabs((p.theta[j] - p.theta[r]) - TWO_PI * (double)q) <= 2e-12;
                }
            if (__syncthreads_and(okf)) P = Pc;
        }
    }
    const int pts_per_surface = p.nalpha * P;
    const int tiles_per_surface = (pts_per_surface + GEO_THREADS - 1) / GEO_THREADS;
    unsigned parity = 0;
    if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();

    // Work = (surface, tile) pairs flattened; every CTA takes one contiguous, equally sized range of them (perfect
    // balance, no tail wave) and re-stages the tables only when its range crosses into the next surface.
    const long long W = (long long)p.ns * tiles_per_surface;
    const long long w_begin = W * blockIdx.x / gridDim.x, w_end = W * (blockIdx.x + 1) / gridDim.x;
    int js = -1;
    double s_val = 0, iota = 1, d_iota = 0, dpds = 0, shat = 0;
    for (long long w = w_begin; w < w_end; ++w) {
        const int js_w = (int)(w / tiles_per_surface);
        const int tile = (int)(w - (long long)js_w * tiles_per_surface);
        if (js_w != js) {
            js = js_w;
            // ---- stage this surface's packed tables in shared memory (TMA bulk copy)
            __syncthreads();                       // everyone is done with the previous surface's tables
            if (tid == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(bar, (unsigned)((n_mn + n_nyq) * sizeof(double)));
                tma_bulk_g2s(s_mn, p.pk_mn + (size_t)js * n_mn, (unsigned)(n_mn * sizeof(double)), bar);
                tma_bulk_g2s(s_nyq, p.pk_nyq + (size_t)js * n_nyq, (unsigned)(n_nyq * sizeof(double)), bar);
            }
            const double* sc = p.scal + (size_t)js * IBS_NSCAL;
            s_val = sc[0]; iota = sc[1]; d_iota = sc[2]; dpds = sc[3]; shat = sc[4];
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        {
            const int pt = tile * GEO_THREADS + tid;
            if (pt >= pts_per_surface) continue;
            const int ja = pt / P, jl = pt - ja * P;
            const double al = p.alpha_per_surface ? p.alpha[(size_t)js * p.nalpha + ja] : p.alpha[ja];
            const double theta_p = p.theta[jl];
            const double phi = p.phi_center + (theta_p - al) / iota;            // utils.py:373

            // cos/sin(k nfp phi), k = 0..NT
            double cn[NT + 1], sn[NT + 1];
            cn[0] = 1.0; sn[0] = 0.0;
            if (NT > 0) {
                sincos((double)p.nfp * phi, &sn[1], &cn[1]);
#pragma unroll
                for (int k = 2; k <= NT; ++k) {
                    cn[k] = fma(cn[k - 1], cn[1], -(sn[k - 1] * sn[1]));
                    sn[k] = fma(sn[k - 1], cn[1], cn[k - 1] * sn[1]);
                }
            }
            // ---- Newton for theta_vmec:  th + sum_m [ sin(m th) A_m - cos(m th) B_m ] = theta_p
            // A_m, B_m: per-thread columns of a shared-memory array [2 m + {0, 1}][thread] (conflict-free), or thread-local
            // arrays when mpol is too large for that
            double AmBm_local[NT1 > 0 ? 2 * MAX_M_NEWTON : 2];
            const bool newton_smem = IBS_GEO_SMEM_NEWTON && NT1 > 0 && p.M1 <= GEO_SMEM_NEWTON_MAX_M;
            double* const ab = newton_smem ? (s_nyq + n_nyq + tid) : AmBm_local;
            const int abs_ = newton_smem ? GEO_THREADS : 1;
#define Am(m) ab[(2 * (m)) * abs_]
#define Bm(m) ab[(2 * (m) + 1) * abs_]
            if (NT1 > 0) {
                for (int m = 0; m < p.M1; ++m) {
                    const double* row = s_mn + (size_t)m * (NT1 + 1) * ROWP_MN + 12;      // (E, O) of the l row
                    double a = row[0], b = 0.0;
#pragma unroll
                    for (int k = 1; k <= NT1; ++k) {
                        const double2 eo = *reinterpret_cast<const double2*>(row + k * ROWP_MN);
                        a = fma(eo.x, cn[k], a);
                        b = fma(eo.y, sn[k], b);
                    }
                    Am(m) = a; Bm(m) = b;
                }
            }
            double th = theta_p;
            int nit = 0; bool ok = false;
            double dprev = 1e300;
            for (nit = 1; nit <= 25; ++nit) {
                double s1, c1;
                sincos(th, &s1, &c1);
                double cm = 1.0, sm = 0.0, fsum = 0.0, dsum = 0.0;
                if constexpr (NT1 == 0) {
                    // axisymmetric tables (n = 0 only): B_m = 0, no toroidal angle; 7 FP64 operations per mode
                    double dm = 0.0;
                    for (int m = 0; m < p.M1; ++m) {
                        const double a = s_mn[(size_t)m * ROW_MN + 6];
                        fsum = fma(sm, a, fsum);
                        dsum = fma(dm * cm, a, dsum);
                        const double cnx = fma(cm, c1, -(sm * s1));
                        sm = fma(sm, c1, cm * s1);
                        cm = cnx;
                        dm += 1.0;
                    }
                } else {
                    for (int m = 0; m < p.M1; ++m) {
                        const double a = Am(m);
                        const double b = Bm(m);
                        fsum = fma(sm, a, fsum); fsum = fma(-cm, b, fsum);
                        const double dm = (double)m;
                        dsum = fma(dm * cm, a, dsum); dsum = fma(dm * sm, b, dsum);
                        const double cnx = fma(cm, c1, -(sm * s1));
                        sm = fma(sm, c1, cm * s1);
                        cm = cnx;
                    }
                }
                const double res = (th + fsum) - theta_p;
                const double dth = res / (1.0 + dsum);
                th -= dth;
                const double ad = fabs(dth), scale_th = fmax(1.0, fabs(th));
                if (ad <= 4.5e-16 * scale_th) { ok = true; break; }
                // quadratic convergence: the error left after this step is ~ ad^3 / dprev^2 -- no confirming iteration
                // once that is below the rounding level
                if (dprev < 1.0 && ad < 1e-3 * dprev) {           // (needs a previous correction, itself already small)
                    const double q = ad / dprev;
                    if (ad * q * q <= 2e-16 * scale_th) { ok = true; break; }
                }
                dprev = ad;
            }
#undef Am
#undef Bm
            // ---- mode sums (utils.py:420-468)
            double s1, c1;
            sincos(th, &s1, &c1);
            double R = 0, R_s = 0, R_t = 0, R_p = 0, Z_s = 0, Z_t = 0, Z_p = 0, L_s = 0, L_t = 0, L_p = 0;
            if (NT1 > 0) {
                double cm = 1.0, sm = 0.0;
                for (int m = 0; m < p.M1; ++m) {
                    const double* row = s_mn + (size_t)m * (NT1 + 1) * ROWP_MN;
                    double A[9], Bv[9];
#pragma unroll
                    for (int j = 0; j < 9; ++j) { A[j] = row[2 * j]; Bv[j] = 0.0; }
#if IBS_GEO_NROWS_DERIVED
                    // The n-weighted rows (n r, n z, n l) are never loaded: with v(-n) the coefficient of -n,
                    //   E_{n v} = k nfp (v(+n) - v(-n)) = k nfp O_v,   O_{n v} = k nfp E_v,
                    // so the pair (E_v, O_v) just loaded feeds FOUR FMAs.  The kernel is bound by the shared-memory data pipe
                    // (one wavefront per loaded double): 12 instead of 18 wavefronts per (m, k) here, 14 instead of 16 below.
                    A[1] = 0.0; A[4] = 0.0; A[7] = 0.0;
#pragma unroll
                    for (int k = 1; k <= NT1; ++k) {
                        const double kn = (double)k * (double)p.nfp;
                        double kc = kn * cn[k], ks = kn * sn[k];
#if IBS_GEO_KC_INLOOP
                        asm volatile("" : "+d"(kc), "+d"(ks));       // (formed here, per m: hoisted they cost 4 NT1 registers)
#endif
#pragma unroll
                        for (int j = 0; j < 9; ++j) {
                            if (j == 1 || j == 4 || j == 7) continue;
                            const double2 eo = *reinterpret_cast<const double2*>(row + k * ROWP_MN + 2 * j);
                            A[j] = fma(eo.x, cn[k], A[j]);
                            Bv[j] = fma(eo.y, sn[k], Bv[j]);
                            if (j == 0 || j == 3 || j == 6) {
                                A[j + 1] = fma(eo.y, kc, A[j + 1]);
                                Bv[j + 1] = fma(eo.x, ks, Bv[j + 1]);
                            }
                        }
                    }
#else
#pragma unroll
                    for (int k = 1; k <= NT1; ++k) {
#pragma unroll
                        for (int j = 0; j < 9; ++j) {
                            const double2 eo = *reinterpret_cast<const double2*>(row + k * ROWP_MN + 2 * j);
                            A[j] = fma(eo.x, cn[k], A[j]);
                            Bv[j] = fma(eo.y, sn[k], Bv[j]);
                        }
                    }
#endif
                    // rows: 0 r, 1 n r, 2 r_s, 3 z, 4 n z, 5 z_s, 6 l, 7 n l, 8 l_s
                    const double dm = (double)m;
                    R += fma(cm, A[0], sm * Bv[0]);
                    R_t = fma(-dm, fma(sm, A[0], -(cm * Bv[0])), R_t);
                    R_p += fma(sm, A[1], -(cm * Bv[1]));
                    R_s += fma(cm, A[2], sm * Bv[2]);
                    Z_t = fma(dm, fma(cm, A[3], sm * Bv[3]), Z_t);
                    Z_p -= fma(cm, A[4], sm * Bv[4]);
                    Z_s += fma(sm, A[5], -(cm * Bv[5]));
                    L_t = fma(dm, fma(cm, A[6], sm * Bv[6]), L_t);
                    L_p -= fma(cm, A[7], sm * Bv[7]);
                    L_s += fma(sm, A[8], -(cm * Bv[8]));
                    const double cnx = fma(cm, c1, -(sm * s1));
                    sm = fma(sm, c1, cm * s1);
                    cm = cnx;
                }
            } else if constexpr (NT1 == 0) {
                // axisymmetric tables: one entry (n = 0) per m, the angle is m theta itself and the n-weighted sums
                // (d/dphi) vanish: 10 FP64 operations per mode + the recurrence
                double cm = 1.0, sm = 0.0, dm = 0.0;
                for (int m = 0; m < p.M1; ++m) {
                    const double* row = s_mn + (size_t)m * ROW_MN;
                    const double2 v0 = *reinterpret_cast<const double2*>(row + 0);   // r, n r (= 0)
                    const double2 v1 = *reinterpret_cast<const double2*>(row + 2);   // r_s, z
                    const double2 v2 = *reinterpret_cast<const double2*>(row + 4);   // n z (= 0), z_s
                    const double2 v3 = *reinterpret_cast<const double2*>(row + 6);   // l, n l (= 0)
                    const double v4 = row[8];                                          // l_s
                    const double msm = dm * sm, mcm = dm * cm;
                    R = fma(v0.x, cm, R);
                    R_t = fma(-v0.x, msm, R_t);
                    R_s = fma(v1.x, cm, R_s);
                    Z_t = fma(v1.y, mcm, Z_t);
                    Z_s = fma(v2.y, sm, Z_s);
                    L_t = fma(v3.x, mcm, L_t);
                    L_s = fma(v4, sm, L_s);
                    const double cnx = fma(cm, c1, -(sm * s1));
                    sm = fma(sm, c1, cm * s1);
                    cm = cnx;
                    dm += 1.0;
                }
            } else {
                double cm = 1.0, sm = 0.0;
                for (int m = 0; m < p.M1; ++m) {
                    const double* row = s_mn + (size_t)m * W1 * ROW_MN;
                    double a0 = 0, a1 = 0, a2 = 0, a3 = 0, a4 = 0, a5 = 0, a6 = 0, a7 = 0, a8 = 0, a9 = 0;
#pragma unroll
                    for (int q = 0; q < W1; ++q) {
                        const int k = q - NT1, ak = k < 0 ? -k : k;
                        double ca, sa;
                        if (k >= 0) angle<1>(cm, sm, cn[ak], sn[ak], ca, sa);
                        else angle<-1>(cm, sm, cn[ak], sn[ak], ca, sa);
                        const double2 v0 = *reinterpret_cast<const double2*>(row + q * ROW_MN + 0);   // r, n r
                        const double2 v1 = *reinterpret_cast<const double2*>(row + q * ROW_MN + 2);   // r_s, z
                        const double2 v2 = *reinterpret_cast<const double2*>(row + q * ROW_MN + 4);   // n z, z_s
                        const double2 v3 = *reinterpret_cast<const double2*>(row + q * ROW_MN + 6);   // l, n l
                        const double v4 = row[q * ROW_MN + 8];                                          // l_s
                        a0 = fma(v0.x, ca, a0);   // sum r cos
                        a1 = fma(v0.x, sa, a1);   // sum r sin
                        a2 = fma(v0.y, sa, a2);   // sum n r sin
                        a3 = fma(v1.x, ca, a3);   // sum r_s cos
                        a4 = fma(v1.y, ca, a4);   // sum z cos
                        a5 = fma(v2.x, ca, a5);   // sum n z cos
                        a6 = fma(v2.y, sa, a6);   // sum z_s sin
                        a7 = fma(v3.x, ca, a7);   // sum l cos
                        a8 = fma(v3.y, ca, a8);   // sum n l cos
                        a9 = fma(v4, sa, a9);     // sum l_s sin
                    }
                    const double dm = (double)m;
                    R += a0; R_t = fma(-dm, a1, R_t); R_p += a2; R_s += a3;
                    Z_t = fma(dm, a4, Z_t); Z_p -= a5; Z_s += a6;
                    L_t = fma(dm, a7, L_t); L_p -= a8; L_s += a9;
                    const double cnx = fma(cm, c1, -(sm * s1));
                    sm = fma(sm, c1, cm * s1);
                    cm = cnx;
                }
            }
            double sqrtg = 0, B = 0, B_s = 0, B_t = 0, B_p = 0, Bsup_p = 0, Bsub_s = 0, Bsub_t = 0, Bsub_p = 0;
            if (NT2 > 0) {
                double cm = 1.0, sm = 0.0;
                for (int m = 0; m < p.M2; ++m) {
                    const double* row = s_nyq + (size_t)m * (NT2 + 1) * ROWP_NYQ;
                    double A[8], Bv[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) { A[j] = row[2 * j]; Bv[j] = 0.0; }
#if IBS_GEO_NROWS_DERIVED
                    A[2] = 0.0;                           // (n b) from (b): see the (R, Z, lambda) set above
#pragma unroll
                    for (int k = 1; k <= NT2; ++k) {
                        const double kn = (double)k * (double)p.nfp;
                        double kc = kn * cn[k], ks = kn * sn[k];
#if IBS_GEO_KC_INLOOP
                        asm volatile("" : "+d"(kc), "+d"(ks));
#endif
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            if (j == 2) continue;
                            const double2 eo = *reinterpret_cast<const double2*>(row + k * ROWP_NYQ + 2 * j);
                            A[j] = fma(eo.x, cn[k], A[j]);
                            Bv[j] = fma(eo.y, sn[k], Bv[j]);
                            if (j == 1) {
                                A[2] = fma(eo.y, kc, A[2]);
                                Bv[2] = fma(eo.x, ks, Bv[2]);
                            }
                        }
                    }
#else
#pragma unroll
                    for (int k = 1; k <= NT2; ++k) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const double2 eo = *reinterpret_cast<const double2*>(row + k * ROWP_NYQ + 2 * j);
                            A[j] = fma(eo.x, cn[k], A[j]);
                            Bv[j] = fma(eo.y, sn[k], Bv[j]);
                        }
                    }
#endif
                    // rows: 0 g, 1 b, 2 n b, 3 b_s, 4 bsupv, 5 bsubs, 6 bsubu, 7 bsubv
                    const double dm = (double)m;
                    sqrtg += fma(cm, A[0], sm * Bv[0]);
                    B += fma(cm, A[1], sm * Bv[1]);
                    B_t = fma(-dm, fma(sm, A[1], -(cm * Bv[1])), B_t);
                    B_p += fma(sm, A[2], -(cm * Bv[2]));
                    B_s += fma(cm, A[3], sm * Bv[3]);
                    Bsup_p += fma(cm, A[4], sm * Bv[4]);
                    Bsub_s += fma(sm, A[5], -(cm * Bv[5]));
                    Bsub_t += fma(cm, A[6], sm * Bv[6]);
                    Bsub_p += fma(cm, A[7], sm * Bv[7]);
                    const double cnx = fma(cm, c1, -(sm * s1));
                    sm = fma(sm, c1, cm * s1);
                    cm = cnx;
                }
            } else if constexpr (NT2 == 0) {
                double cm = 1.0, sm = 0.0, dm = 0.0;
                for (int m = 0; m < p.M2; ++m) {
                    const double* row = s_nyq + (size_t)m * ROW_NYQ;
                    const double2 v0 = *reinterpret_cast<const double2*>(row + 0);  // g, b
                    const double2 v1 = *reinterpret_cast<const double2*>(row + 2);  // n b (= 0), b_s
                    const double2 v2 = *reinterpret_cast<const double2*>(row + 4);  // bsupv, bsubs
                    const double2 v3 = *reinterpret_cast<const double2*>(row + 6);  // bsubu, bsubv
                    sqrtg = fma(v0.x, cm, sqrtg);
                    B = fma(v0.y, cm, B);
                    B_t = fma(-v0.y, dm * sm, B_t);
                    B_s = fma(v1.y, cm, B_s);
                    Bsup_p = fma(v2.x, cm, Bsup_p);
                    Bsub_s = fma(v2.y, sm, Bsub_s);
                    Bsub_t = fma(v3.x, cm, Bsub_t);
                    Bsub_p = fma(v3.y, cm, Bsub_p);
                    const double cnx = fma(cm, c1, -(sm * s1));
                    sm = fma(sm, c1, cm * s1);
                    cm = cnx;
                    dm += 1.0;
                }
            } else {
                double cm = 1.0, sm = 0.0;
                for (int m = 0; m < p.M2; ++m) {
                    const double* row = s_nyq + (size_t)m * W2 * ROW_NYQ;
                    double a0 = 0, a1 = 0, a2 = 0, a3 = 0, a4 = 0, a5 = 0, a6 = 0, a7 = 0, a8 = 0;
#pragma unroll
                    for (int q = 0; q < W2; ++q) {
                        const int k = q - NT2, ak = k < 0 ? -k : k;
                        double ca, sa;
                        if (k >= 0) angle<1>(cm, sm, cn[ak], sn[ak], ca, sa);
                        else angle<-1>(cm, sm, cn[ak], sn[ak], ca, sa);
                        const double2 v0 = *reinterpret_cast<const double2*>(row + q * ROW_NYQ + 0);  // g, b
                        const double2 v1 = *reinterpret_cast<const double2*>(row + q * ROW_NYQ + 2);  // n b, b_s
                        const double2 v2 = *reinterpret_cast<const double2*>(row + q * ROW_NYQ + 4);  // bsupv, bsubs
                        const double2 v3 = *reinterpret_cast<const double2*>(row + q * ROW_NYQ + 6);  // bsubu, bsubv
                        a0 = fma(v0.x, ca, a0);   // sqrt g
                        a1 = fma(v0.y, ca, a1);   // B
                        a2 = fma(v0.y, sa, a2);   // sum b sin
                        a3 = fma(v1.x, sa, a3);   // sum n b sin
                        a4 = fma(v1.y, ca, a4);   // dB/ds
                        a5 = fma(v2.x, ca, a5);   // B^phi
                        a6 = fma(v2.y, sa, a6);   // B_s
                        a7 = fma(v3.x, ca, a7);   // B_theta
                        a8 = fma(v3.y, ca, a8);   // B_phi
                    }
                    const double dm = (double)m;
                    sqrtg += a0; B += a1; B_t = fma(-dm, a2, B_t); B_p += a3; B_s += a4;
                    Bsup_p += a5; Bsub_s += a6; Bsub_t += a7; Bsub_p += a8;
                    const double cnx = fma(cm, c1, -(sm * s1));
                    sm = fma(sm, c1, cm * s1);
                    cm = cnx;
                }
            }
            GeoSums g;
            g.R = R; g.R_s = R_s; g.R_t = R_t; g.R_p = R_p; g.Z_s = Z_s; g.Z_t = Z_t; g.Z_p = Z_p; g.L_s = L_s; g.L_t = L_t; g.L_p = L_p;
            g.sqrtg = sqrtg; g.B = B; g.B_s = B_s; g.B_t = B_t; g.B_p = B_p; g.Bsup_p = Bsup_p; g.Bsub_s = Bsub_s; g.Bsub_t = Bsub_t; g.Bsub_p = Bsub_p;
            if constexpr (NT1 == 0 && NT2 == 0) {
                for (int jf = jl; jf < p.nl; jf += P) {           // the same sums zero, one, two, ... poloidal turns on
                    const double tp = p.theta[jf];
                    geo_point_epilogue(p, g, js, ja, jf, p.phi_center + (tp - al) / iota, th + (tp - theta_p), nit, ok, s_val, iota, d_iota,
                                       dpds, shat);
                }
            } else {
                geo_point_epilogue(p, g, js, ja, jl, phi, th, nit, ok, s_val, iota, d_iota, dpds, shat);
            }
        }
    }
}

// ---- 3-D equilibria: TWO points per thread (any toroidal range; NOT the default) ---------------------------------------
// The paired tables are read with broadcast LDS.128 (E, O): one shared-memory wavefront per FP64 FMA when a thread owns one
// point, and the SM delivers one wavefront per clock against two DFMA warp-instructions -- the one-point kernel runs the
// shared-memory data pipe at 85 % of its peak with the FP64 pipe at 60 % (profiles/geometry_r01c_ncsx): that pipe, not
// latency, is its bound (16 warps / SM at 128 registers are 3-9 % slower).  Here a thread owns P = 2 points, so every
// loaded pair feeds four FMAs, and cos / sin(k nfp phi) are not held as arrays (2 x 28 doubles per point would not fit)
// but advanced inside the k loop by the three-term recurrence
//     cos((k+1) x) = 2 cos x cos(k x) - cos((k-1) x)       (+2 FMAs per (m, k) and point on 18: the price of the registers)
// which also makes the toroidal range a run-time loop bound: one kernel for any |n| / nfp.
// MEASURED (round 2, B200): halving the wavefronts does not pay -- at 254 registers only 8 warps / SM are resident and the
// rolled k loop exposes the load latency: NCSX config 3.51 ms (k loop unrolled by 2: 3.30) against 2.95 for the one-point
// kernel, HBERG 110 / 103 against 92 ms.  It therefore only serves toroidal ranges the templated kernels do not cover
// (|n| / nfp > 18) and IBS_GEO3D=1.
#ifndef IBS_GEO3_UNROLL
#define IBS_GEO3_UNROLL 1
#endif
constexpr int GEO3_P = 2;
constexpr int GEO3_UNROLL = IBS_GEO3_UNROLL;
constexpr int GEO3_THREADS = 128;
constexpr int GEO3_SMEM_NEWTON_MAX_M = 16;     // A_m, B_m of both points live in shared memory when mpol + 1 <= this

struct Geo3Point {
    double theta_p, phi, al, th;
    int ja, jl, nit; bool ok, valid;
};

__global__ void __launch_bounds__(GEO3_THREADS, 2)
geometry3d_kernel(const GeoParams p, const int NT1, const int NT2) {
    constexpr int P = GEO3_P, T = GEO3_THREADS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    double* s_mn = reinterpret_cast<double*>(smem_raw + 16);
    const int n_mn = p.M1 * (NT1 + 1) * ROWP_MN, n_nyq = p.M2 * (NT2 + 1) * ROWP_NYQ;
    double* s_nyq = s_mn + n_mn;
    double* s_ab = s_nyq + n_nyq;                           // [m][A, B][point q][thread]
    const int tid = threadIdx.x;
    const int pts_per_surface = p.nalpha * p.nl;
    const int tiles_per_surface = (pts_per_surface + P * T - 1) / (P * T);
    unsigned parity = 0;
    if (tid == 0) { mbar_init(bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();
    const bool newton_smem = p.M1 <= GEO3_SMEM_NEWTON_MAX_M;
    double ab_local[2 * MAX_M_NEWTON * P];                  // only touched when mpol is too large for the shared array
    double* const ab = newton_smem ? (s_ab + tid) : ab_local;
    const int ab_q = newton_smem ? T : 1, ab_m = newton_smem ? 2 * P * T : 2 * P;       // strides: point, mode
    const int ab_b = newton_smem ? P * T : P;                                              // A -> B

    const long long W = (long long)p.ns * tiles_per_surface;
    const long long w_begin = W * blockIdx.x / gridDim.x, w_end = W * (blockIdx.x + 1) / gridDim.x;
    int js = -1;
    double s_val = 0, iota = 1, d_iota = 0, dpds = 0, shat = 0;
    for (long long w = w_begin; w < w_end; ++w) {
        const int js_w = (int)(w / tiles_per_surface);
        const int tile = (int)(w - (long long)js_w * tiles_per_surface);
        if (js_w != js) {
            js = js_w;
            __syncthreads();                       // everyone is done with the previous surface's tables
            if (tid == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(bar, (unsigned)((n_mn + n_nyq) * sizeof(double)));
                tma_bulk_g2s(s_mn, p.pk_mn + (size_t)js * n_mn, (unsigned)(n_mn * sizeof(double)), bar);
                tma_bulk_g2s(s_nyq, p.pk_nyq + (size_t)js * n_nyq, (unsigned)(n_nyq * sizeof(double)), bar);
            }
            const double* sc = p.scal + (size_t)js * IBS_NSCAL;
            s_val = sc[0]; iota = sc[1]; d_iota = sc[2]; dpds = sc[3]; shat = sc[4];
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        Geo3Point pt[P];
        double c1p[P], s1p[P];                              // cos / sin(nfp phi)
        // ---- per point: angles, n-summed Newton coefficients, theta_vmec
#pragma unroll
        for (int q = 0; q < P; ++q) {
            const int ip = tile * (P * T) + q * T + tid;
            pt[q].valid = ip < pts_per_surface;
            const int ipc = pt[q].valid ? ip : pts_per_surface - 1;          // (an idle slot repeats the last point; nothing is stored)
            pt[q].ja = ipc / p.nl; pt[q].jl = ipc - pt[q].ja * p.nl;
            pt[q].al = p.alpha_per_surface ? p.alpha[(size_t)js * p.nalpha + pt[q].ja] : p.alpha[pt[q].ja];
            pt[q].theta_p = p.theta[pt[q].jl];
            pt[q].phi = p.phi_center + (pt[q].theta_p - pt[q].al) / iota;   // utils.py:373
            sincos((double)p.nfp * pt[q].phi, &s1p[q], &c1p[q]);
            const double tc = 2.0 * c1p[q];
            for (int m = 0; m < p.M1; ++m) {
                const double* row = s_mn + (size_t)m * (NT1 + 1) * ROWP_MN + 12;      // (E, O) of the l row
                double a = row[0], b = 0.0;
                double ck = c1p[q], sk = s1p[q], ckm = 1.0, skm = 0.0;
                for (int k = 1; k <= NT1; ++k) {
                    const double2 eo = *reinterpret_cast<const double2*>(row + k * ROWP_MN);
                    a = fma(eo.x, ck, a);
                    b = fma(eo.y, sk, b);
                    const double cn = fma(tc, ck, -ckm), sn = fma(tc, sk, -skm);
                    ckm = ck; skm = sk; ck = cn; sk = sn;
                }
                ab[m * ab_m + q * ab_q] = a; ab[m * ab_m + ab_b + q * ab_q] = b;
            }
            // Newton:  th + sum_m [ sin(m th) A_m - cos(m th) B_m ] = theta_p   (utils.py:391-416)
            double th = pt[q].theta_p, dprev = 1e300;
            int nit; bool ok = false;
            for (nit = 1; nit <= 25; ++nit) {
                double s1, c1;
                sincos(th, &s1, &c1);
                double cm = 1.0, sm = 0.0, fsum = 0.0, dsum = 0.0;
                for (int m = 0; m < p.M1; ++m) {
                    const double a = ab[m * ab_m + q * ab_q], b = ab[m * ab_m + ab_b + q * ab_q];
                    fsum = fma(sm, a, fsum); fsum = fma(-cm, b, fsum);
                    const double dm = (double)m;
                    dsum = fma(dm * cm, a, dsum); dsum = fma(dm * sm, b, dsum);
                    const double cnx = fma(cm, c1, -(sm * s1));
                    sm = fma(sm, c1, cm * s1);
                    cm = cnx;
                }
                const double res = (th + fsum) - pt[q].theta_p;
                const double dth = res / (1.0 + dsum);
                th -= dth;
                const double ad = fabs(dth), scale_th = fmax(1.0, fabs(th));
                if (ad <= 4.5e-16 * scale_th) { ok = true; break; }
                if (dprev < 1.0 && ad < 1e-3 * dprev) {           // quadratic convergence: see geometry_kernel
                    const double qq = ad / dprev;
                    if (ad * qq * qq <= 2e-16 * scale_th) { ok = true; break; }
                }
                dprev = ad;
            }
            pt[q].th = th; pt[q].nit = nit; pt[q].ok = ok;
        }
        // ---- mode sums of both points against ONE stream of table loads (utils.py:420-468)
        double c1[P], s1[P], tcp[P];
#pragma unroll
        for (int q = 0; q < P; ++q) { sincos(pt[q].th, &s1[q], &c1[q]); tcp[q] = 2.0 * c1p[q]; }
        double R[P], R_s[P], R_t[P], R_p[P], Z_s[P], Z_t[P], Z_p[P], L_s[P], L_t[P], L_p[P];
        {
            double cm[P], sm[P];
#pragma unroll
            for (int q = 0; q < P; ++q) { cm[q] = 1.0; sm[q] = 0.0; R[q] = R_s[q] = R_t[q] = R_p[q] = Z_s[q] = Z_t[q] = Z_p[q] = L_s[q] = L_t[q] = L_p[q] = 0.0; }
            for (int m = 0; m < p.M1; ++m) {
                const double* row = s_mn + (size_t)m * (NT1 + 1) * ROWP_MN;
                double A[P][9], Bv[P][9], ck[P], sk[P], ckm[P], skm[P];
#pragma unroll
                for (int j = 0; j < 9; ++j) {
                    const double a0 = row[2 * j];
#pragma unroll
                    for (int q = 0; q < P; ++q) { A[q][j] = a0; Bv[q][j] = 0.0; }
                }
#pragma unroll
                for (int q = 0; q < P; ++q) { ck[q] = c1p[q]; sk[q] = s1p[q]; ckm[q] = 1.0; skm[q] = 0.0; }
#pragma unroll (GEO3_UNROLL)
                for (int k = 1; k <= NT1; ++k) {
                    const double* rk = row + k * ROWP_MN;
#pragma unroll
                    for (int j = 0; j < 9; ++j) {
                        const double2 eo = *reinterpret_cast<const double2*>(rk + 2 * j);
#pragma unroll
                        for (int q = 0; q < P; ++q) { A[q][j] = fma(eo.x, ck[q], A[q][j]); Bv[q][j] = fma(eo.y, sk[q], Bv[q][j]); }
                    }
#pragma unroll
                    for (int q = 0; q < P; ++q) {
                        const double cn = fma(tcp[q], ck[q], -ckm[q]), sn = fma(tcp[q], sk[q], -skm[q]);
                        ckm[q] = ck[q]; skm[q] = sk[q]; ck[q] = cn; sk[q] = sn;
                    }
                }
                // rows: 0 r, 1 n r, 2 r_s, 3 z, 4 n z, 5 z_s, 6 l, 7 n l, 8 l_s
                const double dm = (double)m;
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    R[q] += fma(cm[q], A[q][0], sm[q] * Bv[q][0]);
                    R_t[q] = fma(-dm, fma(sm[q], A[q][0], -(cm[q] * Bv[q][0])), R_t[q]);
                    R_p[q] += fma(sm[q], A[q][1], -(cm[q] * Bv[q][1]));
                    R_s[q] += fma(cm[q], A[q][2], sm[q] * Bv[q][2]);
                    Z_t[q] = fma(dm, fma(cm[q], A[q][3], sm[q] * Bv[q][3]), Z_t[q]);
                    Z_p[q] -= fma(cm[q], A[q][4], sm[q] * Bv[q][4]);
                    Z_s[q] += fma(sm[q], A[q][5], -(cm[q] * Bv[q][5]));
                    L_t[q] = fma(dm, fma(cm[q], A[q][6], sm[q] * Bv[q][6]), L_t[q]);
                    L_p[q] -= fma(cm[q], A[q][7], sm[q] * Bv[q][7]);
                    L_s[q] += fma(sm[q], A[q][8], -(cm[q] * Bv[q][8]));
                    const double cnx = fma(cm[q], c1[q], -(sm[q] * s1[q]));
                    sm[q] = fma(sm[q], c1[q], cm[q] * s1[q]);
                    cm[q] = cnx;
                }
            }
        }
        double sqrtg[P], B[P], B_s[P], B_t[P], B_p[P], Bsup_p[P], Bsub_s[P], Bsub_t[P], Bsub_p[P];
        {
            double cm[P], sm[P];
#pragma unroll
            for (int q = 0; q < P; ++q) { cm[q] = 1.0; sm[q] = 0.0; sqrtg[q] = B[q] = B_s[q] = B_t[q] = B_p[q] = Bsup_p[q] = Bsub_s[q] = Bsub_t[q] = Bsub_p[q] = 0.0; }
            for (int m = 0; m < p.M2; ++m) {
                const double* row = s_nyq + (size_t)m * (NT2 + 1) * ROWP_NYQ;
                double A[P][8], Bv[P][8], ck[P], sk[P], ckm[P], skm[P];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const double a0 = row[2 * j];
#pragma unroll
                    for (int q = 0; q < P; ++q) { A[q][j] = a0; Bv[q][j] = 0.0; }
                }
#pragma unroll
                for (int q = 0; q < P; ++q) { ck[q] = c1p[q]; sk[q] = s1p[q]; ckm[q] = 1.0; skm[q] = 0.0; }
#pragma unroll (GEO3_UNROLL)
                for (int k = 1; k <= NT2; ++k) {
                    const double* rk = row + k * ROWP_NYQ;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const double2 eo = *reinterpret_cast<const double2*>(rk + 2 * j);
#pragma unroll
                        for (int q = 0; q < P; ++q) { A[q][j] = fma(eo.x, ck[q], A[q][j]); Bv[q][j] = fma(eo.y, sk[q], Bv[q][j]); }
                    }
#pragma unroll
                    for (int q = 0; q < P; ++q) {
                        const double cn = fma(tcp[q], ck[q], -ckm[q]), sn = fma(tcp[q], sk[q], -skm[q]);
                        ckm[q] = ck[q]; skm[q] = sk[q]; ck[q] = cn; sk[q] = sn;
                    }
                }
                // rows: 0 g, 1 b, 2 n b, 3 b_s, 4 bsupv, 5 bsubs, 6 bsubu, 7 bsubv
                const double dm = (double)m;
#pragma unroll
                for (int q = 0; q < P; ++q) {
                    sqrtg[q] += fma(cm[q], A[q][0], sm[q] * Bv[q][0]);
                    B[q] += fma(cm[q], A[q][1], sm[q] * Bv[q][1]);
                    B_t[q] = fma(-dm, fma(sm[q], A[q][1], -(cm[q] * Bv[q][1])), B_t[q]);
                    B_p[q] += fma(sm[q], A[q][2], -(cm[q] * Bv[q][2]));
                    B_s[q] += fma(cm[q], A[q][3], sm[q] * Bv[q][3]);
                    Bsup_p[q] += fma(cm[q], A[q][4], sm[q] * Bv[q][4]);
                    Bsub_s[q] += fma(sm[q], A[q][5], -(cm[q] * Bv[q][5]));
                    Bsub_t[q] += fma(cm[q], A[q][6], sm[q] * Bv[q][6]);
                    Bsub_p[q] += fma(cm[q], A[q][7], sm[q] * Bv[q][7]);
                    const double cnx = fma(cm[q], c1[q], -(sm[q] * s1[q]));
                    sm[q] = fma(sm[q], c1[q], cm[q] * s1[q]);
                    cm[q] = cnx;
                }
            }
        }
        // ---- pointwise algebra and output, one point at a time (utils.py:474-720)
#pragma unroll
        for (int q = 0; q < P; ++q) {
            if (!pt[q].valid) continue;
            GeoSums g;
            g.R = R[q]; g.R_s = R_s[q]; g.R_t = R_t[q]; g.R_p = R_p[q]; g.Z_s = Z_s[q]; g.Z_t = Z_t[q]; g.Z_p = Z_p[q];
            g.L_s = L_s[q]; g.L_t = L_t[q]; g.L_p = L_p[q];
            g.sqrtg = sqrtg[q]; g.B = B[q]; g.B_s = B_s[q]; g.B_t = B_t[q]; g.B_p = B_p[q]; g.Bsup_p = Bsup_p[q];
            g.Bsub_s = Bsub_s[q]; g.Bsub_t = Bsub_t[q]; g.Bsub_p = Bsub_p[q];
            geo_point_epilogue(p, g, js, pt[q].ja, pt[q].jl, pt[q].phi, pt[q].th, pt[q].nit, pt[q].ok, s_val, iota, d_iota, dpds, shat);
        }
    }
}

// dPdrho = -1.0 * 0.5 * mean((cvdrift - gbdrift) * bmag**2)   (ball_scan.py:262); one warp per line.
__global__ void dpdrho_kernel(const double* __restrict__ base, int nlines, int nl, double* __restrict__ out) {
    const int line = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (line >= nlines) return;
    const int lane = threadIdx.x & 31;
    const double* b = base + (size_t)line * IBS_NBASE * nl;
    double acc = 0.0;
    for (int j = lane; j < nl; j += 32) {
        const double bm = b[(size_t)IBS_BASE_BMAG * nl + j];
        acc += __dmul_rn(__dsub_rn(b[(size_t)IBS_BASE_CVDRIFT * nl + j], b[(size_t)IBS_BASE_GBDRIFT * nl + j]), __dmul_rn(bm, bm));
    }
    acc = warp_sum(acc);
    if (lane == 0) out[line] = -1.0 * 0.5 * (acc / (double)nl);
}

// ---- alpha-tangent of K1 (second pass over the packed tables) -------------------------------------------------------------
// alpha enters K1 only through phi = phi_c + (theta_p - alpha) / iota, so at fixed theta_p
//     d/d alpha = phi' d/d phi,   phi' = -1 / iota,   theta_vmec' = theta_phi phi',   theta_phi = -L_p / (1 + L_t)
// (implicit derivative of the converged Newton residual th + lambda(th, phi) = theta_p), and every mode sum moves by
//     S_r' = (T_r theta_phi + P_r) phi',   T_r = d S_r / d theta_vmec (an m-weight),   P_r = d S_r / d phi (an n-weight).
// One thread per point, at the theta_vmec the value pass stored.  With the paired layout (E, O) of ibs_geometry.cu, per
// m and row v: A = sum_k E cos(k nfp phi), B = sum_k O sin(k nfp phi) (k = 0 in A), and their phi-derivatives from the
// same loads, An = sum_k kn O cos, Bn = sum_k kn E sin (kn = k nfp; d A / d phi = -Bn, d B / d phi = An), plus
// Ann = sum_k kn^2 E cos, Bnn = sum_k kn^2 O sin for the rows whose n-weighted sums (R_p, Z_p, L_p, B_p) are outputs.
// A cos-sum is C(A, B) = cm A + sm B, a sin-sum Sn(A, B) = sm A - cm B (cm, sm = cos, sin(m theta_vmec)); then
//     d C / d theta = -m Sn(A, B),  d Sn / d theta = m C(A, B),  d C / d phi = Sn(An, Bn),  d Sn / d phi = -C(An, Bn).
// The axisymmetric tables (dense layout, n = 0 only) are the same code with an empty k loop.  The toroidal range is a
// run-time bound and cos / sin(k nfp phi) advance by the three-term recurrence of geometry3d_kernel: one kernel for every
// shape.  The pointwise algebra is geo_point_epilogue's on D1 (base_point, ibs_geometry_ad.cuh), seeded with S_r' and with
// phi' in sin / cos(phi) and in the secular term (phi - phi_c) iota'.
constexpr int GEO_TAN_THREADS = 128;

__global__ void __launch_bounds__(GEO_TAN_THREADS)
geometry_tangent_kernel(const GeoParams p, const int NT1, const int NT2, const double* __restrict__ thv, double* __restrict__ dbase) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* s_mn = reinterpret_cast<double*>(smem_raw);
    const bool paired = NT1 > 0;                               // geometry_dispatch: NT1 == 0 <=> NT2 == 0 (dense layout)
    const int sm1 = paired ? (NT1 + 1) * ROWP_MN : ROW_MN, sm2 = paired ? (NT2 + 1) * ROWP_NYQ : ROW_NYQ, jst = paired ? 2 : 1;
    const int n_mn = p.M1 * sm1, n_nyq = p.M2 * sm2;
    double* s_nyq = s_mn + n_mn;
    const int tid = threadIdx.x;
    const int pts_per_surface = p.nalpha * p.nl;
    const int tiles_per_surface = (pts_per_surface + GEO_TAN_THREADS - 1) / GEO_TAN_THREADS;
    const long long W = (long long)p.ns * tiles_per_surface;
    const long long w_begin = W * blockIdx.x / gridDim.x, w_end = W * (blockIdx.x + 1) / gridDim.x;
    const double nfp = (double)p.nfp;
    int js = -1;
    double s_val = 0, iota = 1, d_iota = 0, dpds = 0, shat = 0;
    for (long long w = w_begin; w < w_end; ++w) {
        const int js_w = (int)(w / tiles_per_surface);
        const int tile = (int)(w - (long long)js_w * tiles_per_surface);
        if (js_w != js) {
            js = js_w;
            __syncthreads();
            const double* src = p.pk_mn + (size_t)js * n_mn;
            for (int i = tid; i < n_mn; i += GEO_TAN_THREADS) s_mn[i] = src[i];
            src = p.pk_nyq + (size_t)js * n_nyq;
            for (int i = tid; i < n_nyq; i += GEO_TAN_THREADS) s_nyq[i] = src[i];
            const double* sc = p.scal + (size_t)js * IBS_NSCAL;
            s_val = sc[0]; iota = sc[1]; d_iota = sc[2]; dpds = sc[3]; shat = sc[4];
            __syncthreads();
        }
        const int pt = tile * GEO_TAN_THREADS + tid;
        if (pt >= pts_per_surface) continue;
        const int ja = pt / p.nl, jl = pt - ja * p.nl;
        const size_t line = (size_t)js * p.nalpha + ja;
        const double al = p.alpha_per_surface ? p.alpha[(size_t)js * p.nalpha + ja] : p.alpha[ja];
        const double phi = p.phi_center + (p.theta[jl] - al) / iota;            // as in geometry_kernel
        const double th = thv[line * p.nl + jl];
        double s1, c1, s1p = 0.0, c1p = 1.0;
        sincos(th, &s1, &c1);
        if (paired) sincos(nfp * phi, &s1p, &c1p);
        const double tcp = 2.0 * c1p;
        double S[NSUM], T[NSUM], P[NSUM];
#pragma unroll
        for (int r = 0; r < NSUM; ++r) { S[r] = 0.0; T[r] = 0.0; P[r] = 0.0; }
        // ---- (R, Z, lambda) set: rows 0 r, 2 r_s, 3 z, 5 z_s, 6 l, 8 l_s (the n-weighted rows 1, 4, 7 come from the pairs)
        {
            constexpr int RJ[6] = {0, 2, 3, 5, 6, 8};
            double cm = 1.0, sm = 0.0;
            for (int m = 0; m < p.M1; ++m) {
                const double* row = s_mn + (size_t)m * sm1;
                double A[6], Bq[6], An[6], Bn[6], Ann[3], Bnn[3];
#pragma unroll
                for (int i = 0; i < 6; ++i) { A[i] = row[RJ[i] * jst]; Bq[i] = 0.0; An[i] = 0.0; Bn[i] = 0.0; }
#pragma unroll
                for (int i = 0; i < 3; ++i) { Ann[i] = 0.0; Bnn[i] = 0.0; }
                double ck = c1p, sk = s1p, ckm = 1.0, skm = 0.0;
                for (int k = 1; k <= NT1; ++k) {
                    const double kn = (double)k * nfp, kc = kn * ck, ks = kn * sk, kkc = kn * kc, kks = kn * ks;
                    const double* rk = row + k * ROWP_MN;
#pragma unroll
                    for (int i = 0; i < 6; ++i) {
                        const double2 eo = *reinterpret_cast<const double2*>(rk + 2 * RJ[i]);
                        A[i] = fma(eo.x, ck, A[i]); Bq[i] = fma(eo.y, sk, Bq[i]);
                        An[i] = fma(eo.y, kc, An[i]); Bn[i] = fma(eo.x, ks, Bn[i]);
                        if ((i & 1) == 0) { Ann[i / 2] = fma(eo.x, kkc, Ann[i / 2]); Bnn[i / 2] = fma(eo.y, kks, Bnn[i / 2]); }
                    }
                    const double cn = fma(tcp, ck, -ckm), sn = fma(tcp, sk, -skm);
                    ckm = ck; skm = sk; ck = cn; sk = sn;
                }
                const double dm = (double)m, dm2 = dm * dm;
                auto C = [&](double a, double b) { return fma(cm, a, sm * b); };
                auto Sn = [&](double a, double b) { return fma(sm, a, -(cm * b)); };
                // r: R (cos-sum), R_t = dR/dtheta, R_p = dR/dphi
                const double cr = C(A[0], Bq[0]), sr = Sn(A[0], Bq[0]), cnr = C(An[0], Bn[0]), snr = Sn(An[0], Bn[0]);
                S[S_R] += cr;          T[S_R] -= dm * sr;          P[S_R] += snr;
                S[S_Rt] -= dm * sr;    T[S_Rt] -= dm2 * cr;        P[S_Rt] += dm * cnr;
                S[S_Rp] += snr;        T[S_Rp] += dm * cnr;        P[S_Rp] -= C(Ann[0], Bnn[0]);
                S[S_Rs] += C(A[1], Bq[1]);  T[S_Rs] -= dm * Sn(A[1], Bq[1]);  P[S_Rs] += Sn(An[1], Bn[1]);
                // z, lambda: sin-sums; their theta- and phi-derivatives are the outputs
                const double cz = C(A[2], Bq[2]), sz = Sn(A[2], Bq[2]), cnz = C(An[2], Bn[2]), snz = Sn(An[2], Bn[2]);
                S[S_Zt] += dm * cz;    T[S_Zt] -= dm2 * sz;        P[S_Zt] += dm * snz;
                S[S_Zp] -= cnz;        T[S_Zp] += dm * snz;        P[S_Zp] -= Sn(Ann[1], Bnn[1]);
                S[S_Zs] += Sn(A[3], Bq[3]);  T[S_Zs] += dm * C(A[3], Bq[3]);  P[S_Zs] -= C(An[3], Bn[3]);
                const double cl = C(A[4], Bq[4]), sl = Sn(A[4], Bq[4]), cnl = C(An[4], Bn[4]), snl = Sn(An[4], Bn[4]);
                S[S_Lt] += dm * cl;    T[S_Lt] -= dm2 * sl;        P[S_Lt] += dm * snl;
                S[S_Lp] -= cnl;        T[S_Lp] += dm * snl;        P[S_Lp] -= Sn(Ann[2], Bnn[2]);
                S[S_Ls] += Sn(A[5], Bq[5]);  T[S_Ls] += dm * C(A[5], Bq[5]);  P[S_Ls] -= C(An[5], Bn[5]);
                const double cnx = fma(cm, c1, -(sm * s1));
                sm = fma(sm, c1, cm * s1);
                cm = cnx;
            }
        }
        // theta_vmec moves with phi: fold the (R, Z, lambda) derivatives into d S_r / d phi along the field line now (frees P)
        const double th_phi = -S[S_Lp] / (1.0 + S[S_Lt]);                        // d theta_vmec / d phi
#pragma unroll
        for (int r = S_R; r <= S_Lp; ++r) T[r] = fma(T[r], th_phi, P[r]);
        // ---- Nyquist set: rows 0 g, 1 b, 3 b_s, 4 bsupv, 5 bsubs, 6 bsubu, 7 bsubv (row 2, n b, from the b pair)
        {
            constexpr int RJ[7] = {0, 1, 3, 4, 5, 6, 7};
            double cm = 1.0, sm = 0.0;
            for (int m = 0; m < p.M2; ++m) {
                const double* row = s_nyq + (size_t)m * sm2;
                double A[7], Bq[7], An[7], Bn[7], Ann = 0.0, Bnn = 0.0;
#pragma unroll
                for (int i = 0; i < 7; ++i) { A[i] = row[RJ[i] * jst]; Bq[i] = 0.0; An[i] = 0.0; Bn[i] = 0.0; }
                double ck = c1p, sk = s1p, ckm = 1.0, skm = 0.0;
                for (int k = 1; k <= NT2; ++k) {
                    const double kn = (double)k * nfp, kc = kn * ck, ks = kn * sk;
                    const double* rk = row + k * ROWP_NYQ;
#pragma unroll
                    for (int i = 0; i < 7; ++i) {
                        const double2 eo = *reinterpret_cast<const double2*>(rk + 2 * RJ[i]);
                        A[i] = fma(eo.x, ck, A[i]); Bq[i] = fma(eo.y, sk, Bq[i]);
                        An[i] = fma(eo.y, kc, An[i]); Bn[i] = fma(eo.x, ks, Bn[i]);
                        if (i == 1) { Ann = fma(eo.x, kn * kc, Ann); Bnn = fma(eo.y, kn * ks, Bnn); }
                    }
                    const double cn = fma(tcp, ck, -ckm), sn = fma(tcp, sk, -skm);
                    ckm = ck; skm = sk; ck = cn; sk = sn;
                }
                const double dm = (double)m, dm2 = dm * dm;
                auto C = [&](double a, double b) { return fma(cm, a, sm * b); };
                auto Sn = [&](double a, double b) { return fma(sm, a, -(cm * b)); };
                S[S_sqrtg] += C(A[0], Bq[0]);  T[S_sqrtg] -= dm * Sn(A[0], Bq[0]);  P[S_sqrtg] += Sn(An[0], Bn[0]);
                const double cb = C(A[1], Bq[1]), sb = Sn(A[1], Bq[1]), cnb = C(An[1], Bn[1]), snb = Sn(An[1], Bn[1]);
                S[S_B] += cb;          T[S_B] -= dm * sb;          P[S_B] += snb;
                S[S_Bt] -= dm * sb;    T[S_Bt] -= dm2 * cb;        P[S_Bt] += dm * cnb;
                S[S_Bp] += snb;        T[S_Bp] += dm * cnb;        P[S_Bp] -= C(Ann, Bnn);
                S[S_Bs] += C(A[2], Bq[2]);  T[S_Bs] -= dm * Sn(A[2], Bq[2]);  P[S_Bs] += Sn(An[2], Bn[2]);
                S[S_Bsupp] += C(A[3], Bq[3]);  T[S_Bsupp] -= dm * Sn(A[3], Bq[3]);  P[S_Bsupp] += Sn(An[3], Bn[3]);
                S[S_Bsubs] += Sn(A[4], Bq[4]);  T[S_Bsubs] += dm * C(A[4], Bq[4]);  P[S_Bsubs] -= C(An[4], Bn[4]);
                S[S_Bsubt] += C(A[5], Bq[5]);  T[S_Bsubt] -= dm * Sn(A[5], Bq[5]);  P[S_Bsubt] += Sn(An[5], Bn[5]);
                S[S_Bsubp] += C(A[6], Bq[6]);  T[S_Bsubp] -= dm * Sn(A[6], Bq[6]);  P[S_Bsubp] += Sn(An[6], Bn[6]);
                const double cnx = fma(cm, c1, -(sm * s1));
                sm = fma(sm, c1, cm * s1);
                cm = cnx;
            }
        }
        // ---- tangent of the pointwise algebra
        const double dphi = -1.0 / iota;                                        // d phi / d alpha
#pragma unroll
        for (int r = S_sqrtg; r < NSUM; ++r) T[r] = fma(T[r], th_phi, P[r]);
        D1 Sd[NSUM];
#pragma unroll
        for (int r = 0; r < NSUM; ++r) Sd[r] = D1(S[r], T[r] * dphi);
        PointConst<D1> k;
        double sp, cp;
        sincos(phi, &sp, &cp);
        k.sp = D1(sp, cp * dphi); k.cp = D1(cp, -sp * dphi); k.dphi = D1(phi - p.phi_center, dphi);
        k.iota = D1(iota); k.d_iota = D1(d_iota); k.dpds = D1(dpds); k.shat = D1(shat); k.s_val = D1(s_val);
        k.psi_e = D1(p.psi_e); k.L_ref = D1(p.L_ref);
        k.th0 = k.dP = k.sg = k.sc = k.sf = k.qw = 0.0;
        D1 o[IBS_NBASE];
        base_point(Sd, k, o);
        double* d = dbase + line * IBS_NBASE * p.nl + jl;
#pragma unroll
        for (int r = 0; r < IBS_NBASE; ++r) d[(size_t)r * p.nl] = o[r].d;
    }
}

// d(dPdrho) / d alpha = -0.5 mean( d[(cvdrift - gbdrift) bmag^2] / d alpha ); one warp per line, as dpdrho_kernel
__global__ void ddpdrho_kernel(const double* __restrict__ base, const double* __restrict__ dbase, int nlines, int nl,
                               double* __restrict__ out) {
    const int line = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (line >= nlines) return;
    const int lane = threadIdx.x & 31;
    const double* b = base + (size_t)line * IBS_NBASE * nl;
    const double* db = dbase + (size_t)line * IBS_NBASE * nl;
    double acc = 0.0;
    for (int j = lane; j < nl; j += 32) {
        const double bm = b[(size_t)IBS_BASE_BMAG * nl + j];
        const double cg = b[(size_t)IBS_BASE_CVDRIFT * nl + j] - b[(size_t)IBS_BASE_GBDRIFT * nl + j];
        const double dcg = db[(size_t)IBS_BASE_CVDRIFT * nl + j] - db[(size_t)IBS_BASE_GBDRIFT * nl + j];
        acc += fma(dcg, bm * bm, 2.0 * cg * bm * db[(size_t)IBS_BASE_BMAG * nl + j]);
    }
    acc = warp_sum(acc);
    if (lane == 0) out[line] = -0.5 * (acc / (double)nl);
}

// ---- host side ------------------------------------------------------------------------------------------------
template <int NT1, int NT2>
static int launch_geometry(const GeoParams& p, cudaStream_t st) {
    auto kern = geometry_kernel<NT1, NT2>;
    constexpr int GEO_THREADS = GeoThreads<NT1>::value;
    const size_t e_mn = (NT1 > 0) ? (size_t)(NT1 + 1) * ROWP_MN : (size_t)ROW_MN, e_nyq = (NT2 > 0) ? (size_t)(NT2 + 1) * ROWP_NYQ : (size_t)ROW_NYQ;
    const bool newton_smem = IBS_GEO_SMEM_NEWTON && NT1 > 0 && p.M1 <= GEO_SMEM_NEWTON_MAX_M;
    const size_t smem = 16 + ((size_t)p.M1 * e_mn + (size_t)p.M2 * e_nyq + (newton_smem ? (size_t)2 * p.M1 * GEO_THREADS : 0)) * sizeof(double);
    if (smem > 220 * 1024) { set_error("Fourier tables of one surface do not fit in shared memory"); return IBS_ERR_UNSUPPORTED; }
    static bool configured[IBS_MAX_DEVICES] = {false};     // per instantiation and per device (the attribute is per device)
    const int dslot = current_device_slot();
    if (!configured[dslot]) {
        IBS_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        configured[dslot] = true;
    }
    int per_sm = 0;
    IBS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GEO_THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    const int tiles = (p.nalpha * p.nl + GEO_THREADS - 1) / GEO_THREADS;
    const long long slots = (long long)num_sms() * per_sm;
    // persistent 1-D grid: one CTA per resident slot (or per tile when there is less work than that)
    const long long W = (long long)p.ns * tiles;
    const int grid = (int)(W < slots ? W : slots);
    kern<<<grid, GEO_THREADS, smem, st>>>(p);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

static int launch_geometry3d(const GeoParams& p, int NT1, int NT2, cudaStream_t st) {
    const bool newton_smem = p.M1 <= GEO3_SMEM_NEWTON_MAX_M;
    const size_t smem = 16 + ((size_t)p.M1 * (NT1 + 1) * ROWP_MN + (size_t)p.M2 * (NT2 + 1) * ROWP_NYQ +
                              (newton_smem ? (size_t)2 * p.M1 * GEO3_P * GEO3_THREADS : 0)) * sizeof(double);
    if (smem > 220 * 1024) { set_error("Fourier tables of one surface do not fit in shared memory"); return IBS_ERR_UNSUPPORTED; }
    static bool configured[IBS_MAX_DEVICES] = {false};
    const int dslot = current_device_slot();
    if (!configured[dslot]) {
        IBS_CUDA_CHECK(cudaFuncSetAttribute(geometry3d_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        configured[dslot] = true;
    }
    int per_sm = 0;
    IBS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, geometry3d_kernel, GEO3_THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    const int tiles = (p.nalpha * p.nl + GEO3_P * GEO3_THREADS - 1) / (GEO3_P * GEO3_THREADS);
    const long long slots = (long long)num_sms() * per_sm, W = (long long)p.ns * tiles;
    const int grid = (int)(W < slots ? W : slots);
    geometry3d_kernel<<<grid, GEO3_THREADS, smem, st>>>(p, NT1, NT2);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

static int launch_geometry_tangent(const GeoParams& p, int NT1, int NT2, const double* thv, double* dbase, cudaStream_t st) {
    const size_t smem = (NT1 > 0 ? (size_t)p.M1 * (NT1 + 1) * ROWP_MN + (size_t)p.M2 * (NT2 + 1) * ROWP_NYQ
                                 : (size_t)p.M1 * ROW_MN + (size_t)p.M2 * ROW_NYQ) * sizeof(double);
    if (smem > 220 * 1024) { set_error("Fourier tables of one surface do not fit in shared memory"); return IBS_ERR_UNSUPPORTED; }
    static bool configured[IBS_MAX_DEVICES] = {false};
    const int dslot = current_device_slot();
    if (!configured[dslot]) {
        IBS_CUDA_CHECK(cudaFuncSetAttribute(geometry_tangent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        configured[dslot] = true;
    }
    int per_sm = 0;
    IBS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, geometry_tangent_kernel, GEO_TAN_THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    const int tiles = (p.nalpha * p.nl + GEO_TAN_THREADS - 1) / GEO_TAN_THREADS;
    const long long slots = (long long)num_sms() * per_sm, W = (long long)p.ns * tiles;
    const int grid = (int)(W < slots ? W : slots);
    geometry_tangent_kernel<<<grid, GEO_TAN_THREADS, smem, st>>>(p, NT1, NT2, thv, dbase);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

static int gcd_int(int a, int b) { a = std::abs(a); b = std::abs(b); while (b) { int t = a % b; a = b; b = t; } return a; }

// K1, and with dbase_out its alpha-tangent: the value kernel runs unchanged (so its outputs are those of ibs_geometry_batch
// bit for bit), then geometry_tangent_kernel on the same packed tables at the theta_vmec it stored
static int geometry_run(const double* tab_mn, const double* tab_nyq, const double* scal,
                        const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                        int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                        const double* alpha, int nalpha, int alpha_per_surface, const double* theta, int nl,
                        double phi_center, double* base_out, double* dPdrho_out, double* theta_vmec_out,
                        int* info_out, double* dbase_out, double* ddPdrho_out, cudaStream_t st) {
    // ---- mode bookkeeping (host): toroidal stride, extents, dense-grid index of every mode
    int nfp = 0, mmax1 = 0, mmax2 = 0;
    for (int k = 0; k < mnmax; ++k) { nfp = gcd_int(nfp, (int)std::lround(xn[k])); mmax1 = std::max(mmax1, (int)std::lround(xm[k])); }
    for (int k = 0; k < mnmax_nyq; ++k) { nfp = gcd_int(nfp, (int)std::lround(xn_nyq[k])); mmax2 = std::max(mmax2, (int)std::lround(xm_nyq[k])); }
    if (nfp == 0) nfp = 1;
    int nt1 = 0, nt2 = 0;
    std::vector<int> h_idx(2 * (size_t)(mnmax + mnmax_nyq));
    int* m1 = h_idx.data(); int* n1 = m1 + mnmax; int* m2 = n1 + mnmax; int* n2 = m2 + mnmax_nyq;
    for (int k = 0; k < mnmax; ++k) {
        m1[k] = (int)std::lround(xm[k]); n1[k] = (int)std::lround(xn[k]) / nfp;
        IBS_REQUIRE(m1[k] >= 0 && std::fabs(xm[k] - m1[k]) < 1e-9 && std::fabs(xn[k] - (double)n1[k] * nfp) < 1e-9, "non-integer mode numbers");
        nt1 = std::max(nt1, std::abs(n1[k]));
    }
    for (int k = 0; k < mnmax_nyq; ++k) {
        m2[k] = (int)std::lround(xm_nyq[k]); n2[k] = (int)std::lround(xn_nyq[k]) / nfp;
        IBS_REQUIRE(m2[k] >= 0 && std::fabs(xm_nyq[k] - m2[k]) < 1e-9 && std::fabs(xn_nyq[k] - (double)n2[k] * nfp) < 1e-9, "non-integer mode numbers");
        nt2 = std::max(nt2, std::abs(n2[k]));
    }
    // 3-D tables: the one-point-per-thread instantiations (|n| / nfp <= 18) are the default; the two-points-per-thread kernel
    // takes the toroidal ranges as run-time loop bounds, so it serves any wider range (and IBS_GEO3D=1 forces it, for comparison)
    bool use3d = (nt1 > 16 || nt2 > 18);
    if (const char* e = std::getenv("IBS_GEO3D")) { if (std::atoi(e) != 0 && (nt1 > 0 || nt2 > 0)) use3d = true; }
    int NT1, NT2;
    if (nt1 == 0 && nt2 == 0) { NT1 = 0; NT2 = 0; }
    else if (use3d) { NT1 = std::max(nt1, 1); NT2 = std::max(nt2, 1); }
    else if (nt1 <= 6 && nt2 <= 8) { NT1 = 6; NT2 = 8; }
    else if (nt1 <= 11 && nt2 <= 13) { NT1 = 11; NT2 = 13; }
    else { NT1 = 16; NT2 = 18; }
    const int M1 = mmax1 + 1, M2 = mmax2 + 1, W1 = 2 * NT1 + 1, W2 = 2 * NT2 + 1;
    if (NT1 > 0 && M1 > MAX_M_NEWTON) { set_error("mpol too large for a 3-D equilibrium"); return IBS_ERR_UNSUPPORTED; }

    // ---- workspace: packed tables (stream-ordered allocation) + cached device copy of the mode indices
    const size_t n_mn = (size_t)ns * M1 * (NT1 > 0 ? (size_t)(NT1 + 1) * ROWP_MN : (size_t)W1 * ROW_MN);
    const size_t n_nyq = (size_t)ns * M2 * (NT2 > 0 ? (size_t)(NT2 + 1) * ROWP_NYQ : (size_t)W2 * ROW_NYQ);
    double* pk = nullptr; int* d_idx = nullptr;
    {
        // The mode layout of an equilibrium family never changes between calls: keep the last one on
        // the device so steady-state calls issue no host->device copy and no host synchronisation.
        // One slot per device (a process may drive several GPUs); a replaced layout is freed after a device-wide
        // synchronisation, because launches on other streams may still read it.
        struct ModeCache { std::vector<int> host; int* dev = nullptr; };
        static std::mutex mu;
        static ModeCache cache[IBS_MAX_DEVICES];
        std::lock_guard<std::mutex> lk(mu);
        ModeCache& mc = cache[current_device_slot()];
        if (!(mc.dev && mc.host == h_idx)) {
            if (mc.dev) { IBS_CUDA_CHECK(cudaDeviceSynchronize()); cudaFree(mc.dev); mc.dev = nullptr; mc.host.clear(); }
            IBS_CUDA_CHECK(cudaMalloc((void**)&mc.dev, h_idx.size() * sizeof(int)));
            IBS_CUDA_CHECK(cudaMemcpy(mc.dev, h_idx.data(), h_idx.size() * sizeof(int), cudaMemcpyHostToDevice));
            mc.host = h_idx;
        }
        d_idx = mc.dev;
    }
    keep_pool_cached();
    // the tangent pass reads theta_vmec: a scratch copy after the tables when the caller does not want it
    const size_t n_thv = (dbase_out && !theta_vmec_out) ? (size_t)ns * nalpha * nl : 0;
    IBS_CUDA_CHECK(cudaMallocAsync((void**)&pk, (n_mn + n_nyq + n_thv) * sizeof(double), st));
    IBS_CUDA_CHECK(cudaMemsetAsync(pk, 0, (n_mn + n_nyq) * sizeof(double), st));
    if (n_thv) theta_vmec_out = pk + n_mn + n_nyq;
    pack_mn_kernel<<<dim3(ns, (mnmax + 127) / 128), 128, 0, st>>>(tab_mn, d_idx, d_idx + mnmax, ns, mnmax, M1, W1, NT1, nfp, pk);
    pack_nyq_kernel<<<dim3(ns, (mnmax_nyq + 127) / 128), 128, 0, st>>>(tab_nyq, d_idx + 2 * mnmax, d_idx + 2 * mnmax + mnmax_nyq, ns,
                                                                     mnmax_nyq, M2, W2, NT2, nfp, pk + n_mn);
    IBS_CUDA_CHECK(cudaGetLastError());

    GeoParams p;
    p.pk_mn = pk; p.pk_nyq = pk + n_mn; p.scal = scal;
    p.alpha = alpha; p.nalpha = nalpha; p.alpha_per_surface = alpha_per_surface;
    p.theta = theta; p.nl = nl; p.ns = ns; p.M1 = M1; p.M2 = M2; p.nfp = nfp;
    p.phi_center = phi_center; p.psi_e = -phiedge / (2.0 * 3.141592653589793); p.L_ref = aminor_p;
    p.base_out = base_out; p.theta_vmec_out = theta_vmec_out; p.info_out = info_out;
    { const char* e = std::getenv("IBS_GEO_FOLD"); p.fold = !(e && e[0] == '0'); }
    if (info_out) IBS_CUDA_CHECK(cudaMemsetAsync(info_out, 0, (size_t)ns * nalpha * sizeof(int), st));
    int rc;
    if (NT1 == 0) rc = launch_geometry<0, 0>(p, st);
    else if (use3d) rc = launch_geometry3d(p, NT1, NT2, st);
    else if (NT1 == 6) rc = launch_geometry<6, 8>(p, st);
    else if (NT1 == 11) rc = launch_geometry<11, 13>(p, st);
    else rc = launch_geometry<16, 18>(p, st);
    if (rc == IBS_OK && dPdrho_out) {
        const int nlines = ns * nalpha;
        dpdrho_kernel<<<(nlines + 3) / 4, 128, 0, st>>>(base_out, nlines, nl, dPdrho_out);
        if (cudaGetLastError() != cudaSuccess) rc = IBS_ERR_CUDA;
    }
    if (rc == IBS_OK && dbase_out) {
        rc = launch_geometry_tangent(p, NT1, NT2, theta_vmec_out, dbase_out, st);
        if (rc == IBS_OK && ddPdrho_out) {
            const int nlines = ns * nalpha;
            ddpdrho_kernel<<<(nlines + 3) / 4, 128, 0, st>>>(base_out, dbase_out, nlines, nl, ddPdrho_out);
            if (cudaGetLastError() != cudaSuccess) rc = IBS_ERR_CUDA;
        }
    }
    cudaFreeAsync(pk, st);
    return rc;
}

int geometry_dispatch(const double* tab_mn, const double* tab_nyq, const double* scal,
                      const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                      int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                      const double* alpha, int nalpha, int alpha_per_surface, const double* theta, int nl,
                      double phi_center, double* base_out, double* dPdrho_out, double* theta_vmec_out,
                      int* info_out, cudaStream_t st) {
    return geometry_run(tab_mn, tab_nyq, scal, xm, xn, xm_nyq, xn_nyq, ns, mnmax, mnmax_nyq, phiedge, aminor_p, alpha, nalpha,
                        alpha_per_surface, theta, nl, phi_center, base_out, dPdrho_out, theta_vmec_out, info_out, nullptr, nullptr, st);
}

int geometry_tangent_dispatch(const double* tab_mn, const double* tab_nyq, const double* scal,
                              const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                              int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                              const double* alpha, int nalpha, int alpha_per_surface, const double* theta, int nl,
                              double phi_center, double* base_out, double* dPdrho_out, double* dbase_out, double* ddPdrho_out,
                              double* theta_vmec_out, int* info_out, cudaStream_t st) {
    return geometry_run(tab_mn, tab_nyq, scal, xm, xn, xm_nyq, xn_nyq, ns, mnmax, mnmax_nyq, phiedge, aminor_p, alpha, nalpha,
                        alpha_per_surface, theta, nl, phi_center, base_out, dPdrho_out, theta_vmec_out, info_out, dbase_out,
                        ddPdrho_out, st);
}

}  // namespace ibs
