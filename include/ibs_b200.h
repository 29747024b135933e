/* ibs_b200.h -- C ABI of the B200-native ideal-ballooning hot path.
 *
 * The reference (rahulgaur104/ideal-ballooning-solver) is pure Python and has no FFI layer; the
 * boundary this library sits behind is the set of Python call signatures that ball_scan.py reaches
 * through `from utils import *` (ball_scan.py:19).  Each entry point below names the reference
 * interface it replaces (file:line under /root/reference).  INTEGRATION.md shows the ctypes stub a
 * maintainer would add on the reference side.
 *
 * Conventions
 *   - all arrays are fp64, row-major, caller-allocated; pointers are DEVICE pointers unless the
 *     function name ends in `_host`;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) and does not synchronise
 *     the host.  State kept between calls: the thread-local error string and, PER DEVICE and behind a
 *     mutex, caches that never change results (kernel attributes set once, the device copy of the
 *     last Fourier-mode layout, the streams/events of ibs_scan_host, the memory-pool threshold); one
 *     process may therefore drive several GPUs (cudaSetDevice before the call);
 *   - return value 0 = OK, non-zero = error (see ibs_last_error());
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 *
 * Grid convention: N = number of theta points of a field line (the reference's `ntheta`,
 * ball_scan.py:203-208), M = N-2 interior unknowns (Dirichlet ends, utils.py:1607-1608).
 */
#ifndef IBS_B200_H
#define IBS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define IBS_OK 0
#define IBS_ERR_INVALID 1   /* bad argument                                   */
#define IBS_ERR_CUDA 2      /* CUDA runtime error (message in ibs_last_error) */
#define IBS_ERR_UNSUPPORTED 3

/* Layout of the per-field-line "base" arrays produced by ibs_geometry_batch and consumed by the
 * solver/adjoint entry points: base[line][IBS_NBASE][N].  These are exactly the eight quantities the
 * reference's hot path reads from the vmec_fieldlines Struct (ball_scan.py:254-261, utils.py:1649-1656). */
#define IBS_BASE_BMAG 0
#define IBS_BASE_GRADPAR 1     /* gradpar_theta_pest */
#define IBS_BASE_CVDRIFT 2
#define IBS_BASE_CVDRIFT0 3
#define IBS_BASE_GDS2 4
#define IBS_BASE_GDS21 5
#define IBS_BASE_GDS22 6
#define IBS_BASE_GBDRIFT 7
#define IBS_NBASE 8

/* rows of the per-surface Fourier tables (utils.py:318-357) */
#define IBS_TAB_MN_ROWS 6      /* rmnc zmns lmns d_rmnc_d_s d_zmns_d_s d_lmns_d_s               */
#define IBS_TAB_NYQ_ROWS 7     /* gmnc bmnc d_bmnc_d_s bsupvmnc bsubsmns bsubumnc bsubvmnc      */
#define IBS_NSCAL 8            /* s iota d_iota_d_s d_pressure_d_s shat pressure (2 spare)      */

/* bits of the per-solve info word written by the solver: info = iterations | flags << 16 */
#define IBS_FLAG_NOT_CONVERGED 1   /* iteration cap hit                                          */
#define IBS_FLAG_BAD_INPUT 2       /* non-finite input, or g <= 0 / f <= 0 somewhere            */
#define IBS_FLAG_SIGMA_NOT_MAX 4   /* eigenvalue nearest sigma (ARPACK semantics) is not lambda_max */

int ibs_version(void);
const char* ibs_last_error(void);
/* number of SMs / compute capability of the current device (0 on success) */
int ibs_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* Measurement aid (bench.py): launches independent DFMA chains on every SM (32 warps per SM, 8 chains per thread) so
 * that the caller can time the device's FP64 FMA peak with CUDA events -- the denominator of the FP64-pipe rooflines of
 * K1 and K2+K3.  scratch [>= 4 * SMs * 256] doubles (device); *fma_count_out (host) = FMAs one launch executes.       */
int ibs_fp64_probe(int iters, double* scratch, long long scratch_len, double* fma_count_out, void* stream);

/* ---- K1: field-line geometry ------------------------------------------------------------------
 * Batched vmec_fieldlines(vs, s, alpha, theta1d=theta) (utils.py:161-864) restricted to the eight
 * arrays the ballooning path reads, for ns surfaces x nalpha field lines x nl points:
 * theta_vmec root solve (utils.py:391-416), the 19 Fourier mode sums (utils.py:420-468), the
 * Cartesian dual basis / drifts (utils.py:474-658) and the GS2 normalisations (utils.py:662-720).
 * Also forms dPdrho = -0.5*mean((cvdrift-gbdrift)*bmag^2) per line (ball_scan.py:262).
 *   tab_mn  [ns][6][mnmax], tab_nyq [ns][7][mnmax_nyq], scal [ns][8]: per-surface tables
 *   xm,xn [mnmax], xm_nyq,xn_nyq [mnmax_nyq]: mode numbers (xn already multiplied by nfp) -- HOST pointers
 *          (metadata: the library derives the dense (m, n) layout from them and caches it on the device)
 *   alpha: [nalpha] shared by all surfaces (alpha_per_surface = 0) or [ns][nalpha] (= 1)
 *   theta [nl]: theta_pest grid; phi = phi_center + (theta - alpha)/iota (utils.py:373)
 *   base_out [ns*nalpha][8][nl]; dPdrho_out [ns*nalpha]; theta_vmec_out [ns*nalpha][nl] or NULL;
 *   info_out [ns*nalpha] or NULL: max Newton iterations used | (not converged) << 16              */
int ibs_geometry_batch(const double* tab_mn, const double* tab_nyq, const double* scal,
                       const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                       int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                       const double* alpha, int nalpha, int alpha_per_surface,
                       const double* theta, int nl, double phi_center,
                       double* base_out, double* dPdrho_out, double* theta_vmec_out, int* info_out,
                       void* stream);

/* K1 and its exact alpha-derivative.  Same arguments and value outputs as ibs_geometry_batch (base_out, dPdrho_out,
 * theta_vmec_out and info_out are bit-identical to its), plus the tangent d/dalpha at fixed theta_pest of every base
 * array and of dPdrho.  alpha enters only through phi = phi_center + (theta - alpha)/iota; theta_vmec moves with it by the
 * implicit derivative of its root equation.  A second pass over the packed tables after the value kernel.
 *   dbase_out [ns*nalpha][8][nl] (required); ddPdrho_out [ns*nalpha] or NULL.                                       */
int ibs_geometry_tangent_batch(const double* tab_mn, const double* tab_nyq, const double* scal,
                               const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                               int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                               const double* alpha, int nalpha, int alpha_per_surface,
                               const double* theta, int nl, double phi_center,
                               double* base_out, double* dPdrho_out, double* dbase_out, double* ddPdrho_out,
                               double* theta_vmec_out, int* info_out, void* stream);

/* Full-output geometry: every per-point array of the Struct returned by vmec_fieldlines (utils.py:723-864) and by
 * vmec_fieldlines_axisym (utils.py:872-1542) -- the ~70 arrays gyrokinetic-geometry consumers read beyond the eight of
 * the ballooning path.  Not a hot kernel (direct mode sums; any mode list).  ALL pointers are device pointers.
 *   tab_mn [ns][6][mnmax], tab_nyq [ns][7][mnmax_nyq] as above, bsupumnc [ns][mnmax_nyq] (the one table K1 does not
 *   need), scal [ns][8]; xm, xn [mnmax], xm_nyq, xn_nyq [mnmax_nyq]; alpha [nalpha]; grid [nl];
 *   mode 0: grid = theta_pest (vmec_fieldlines(theta1d=...)); mode 1: grid = phi (vmec_fieldlines(phi1d=...), utils.py:364-369);
 *   mode 2: grid = theta_vmec, no root solve, the mode sums use theta_vmec + theta_shift and phi = 0, then
 *           theta_pest = theta_vmec + lambda (vmec_fieldlines_axisym, utils.py:972-1046); zero_xn_nyq as utils.py:913;
 *   out [ns*nalpha][ibs_geometry_full_nfields()][nl] in the field order of csrc/ibs_geometry_full.cu (mirrored by
 *   reference_api.FULL_FIELDS); info_out [ns*nalpha] or NULL: Newton iterations | (not converged) << 16.              */
int ibs_geometry_full_nfields(void);
int ibs_geometry_full(const double* tab_mn, const double* tab_nyq, const double* bsupumnc, const double* scal,
                      const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                      int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                      const double* alpha, int nalpha, const double* grid, int nl, int mode, double theta_shift,
                      int zero_xn_nyq, double phi_center, double* out, int* info_out, void* stream);

/* Reverse mode of K1: d(lambda) / d(Fourier table coefficient) for ns field lines, one per surface (row f3: replaces the
 * ndofs + 1 perturbed-equilibrium scans of sims_runner_NCSX.py:245-262 by ONE scan + this call + dot products with the
 * table perturbations).  Chains the Hellmann-Feynman sensitivities of ibs_adjoint_sensitivities (utils.py:1676-1680) through
 * g, c, f (utils.py:1560-1562), the theta0 shift (ball_scan.py:267-268), dPdrho (ball_scan.py:262), the pointwise geometry
 * (utils.py:474-720), the theta_vmec root (utils.py:391-416) and the mode sums (utils.py:432-468), at fixed iota(s), p'(s)
 * (ibs_geometry_adjoint_scal below adds the derivatives with respect to those scalars).
 *   tables / modes as ibs_geometry_full (ALL device pointers); alpha [ns], theta0 [ns], dPdrho [ns]: the line of each surface;
 *   dlam_dg, dlam_dc, dlam_df [ns][nl]; Q [ns] = sum_j dlam_dc_j c_j / (-dPdrho);
 *   grad_mn_out [ns][6][mnmax], grad_nyq_out [ns][7][mnmax_nyq]: d lambda / d tab_mn, d lambda / d tab_nyq.              */
int ibs_geometry_adjoint(const double* tab_mn, const double* tab_nyq, const double* scal,
                         const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                         int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                         const double* alpha, const double* theta, int nl, double phi_center,
                         const double* theta0, const double* dPdrho, const double* dlam_dg, const double* dlam_dc,
                         const double* dlam_df, const double* Q, double* grad_mn_out, double* grad_nyq_out, void* stream);

/* The same reverse mode, plus the derivative of each surface's lambda with respect to the scalar inputs K1 reads.  Arguments
 * as ibs_geometry_adjoint (same order; grad_mn_out and grad_nyq_out are bit-identical to its outputs), then
 *   grad_scal_out [ns][8]: d lambda / d scal[js][k] in the column order of scal (s, iota, d_iota_d_s, d_pressure_d_s, shat;
 *          columns 5-7 -- pressure and the two spares -- are not read by K1 and are exactly 0);
 *   grad_glob_out [ns][2]: (d lambda / d phiedge, d lambda / d Aminor_p) of each surface's lambda.
 * Each is a partial derivative per column with the other columns held fixed: iota, iota' and shat = -2 s iota' / iota are
 * separate inputs of K1.  A consistent perturbation of an equilibrium moves all three; the dot product of these gradients
 * with the actual column differences then gives the total first-order change.  One fixed-order sum per surface: two calls
 * on the same input give identical bits.                                                                                 */
int ibs_geometry_adjoint_scal(const double* tab_mn, const double* tab_nyq, const double* scal,
                              const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                              int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                              const double* alpha, const double* theta, int nl, double phi_center,
                              const double* theta0, const double* dPdrho, const double* dlam_dg, const double* dlam_dc,
                              const double* dlam_df, const double* Q, double* grad_mn_out, double* grad_nyq_out,
                              double* grad_scal_out, double* grad_glob_out, void* stream);

/* ---- K2+K3: discretisation + lambda_max + eigenfunction -------------------------------------------
 * Batched gamma_ball_full (utils.py:1550-1624): g, c, f -> half-grid g, second-order finite
 * differences, Dirichlet ends (utils.py:1564-1592) -> largest eigenvalue and eigenvector of
 * A = F^-1 (D g D + c) -> X = v / max|v| (utils.py:1605), dX stencil (utils.py:1610-1616), Simpson
 * Rayleigh quotient gam = int(-g dX^2 + c X^2) / int(f X^2) (utils.py:1618-1621).
 *   g, c, f [nsolve][N] on a uniform theta grid of spacing h (the reference's np.diff(theta_half)[2])
 *   lam0   [nsolve] or NULL: optional starting shifts (any value is safe)
 *   sigma  [nsolve] or NULL: if given, IBS_FLAG_SIGMA_NOT_MAX is raised when ARPACK's
 *          "eigenvalue nearest sigma" (utils.py:1597) would not be lambda_max
 *   chain_len: > 1 = runs of chain_len consecutive solves are processed back to back by one CTA and each
 *          is warm-started from its predecessor's eigenvalue -- the batched form of the start-vector chain
 *          of ball_scan.py:265-274 (in the base-array entry point a chain never crosses field lines, except when
 *          nth0 == 1, i.e. an alpha scan with one solve per line, where consecutive lines are chained);
 *          <= 1 = independent solves.  Either way every solve is converged to the same tolerance.
 *   lam_out [nsolve]: the reference's returned `gam`; lam_matrix_out [nsolve] or NULL: lambda_max of
 *          the pencil itself; X_out, dX_out [nsolve][N] or NULL (X >= 0, max X = 1);
 *   info_out [nsolve] or NULL.                                                                        */
int ibs_solve_gcf_batch(const double* g, const double* c, const double* f, int nsolve, int N, double h,
                        const double* lam0, const double* sigma, int chain_len,
                        double* lam_out, double* lam_matrix_out, double* X_out, double* dX_out,
                        int* info_out, void* stream);

/* Same solve, but the coefficients are formed on the fly from the base arrays of a field line
 * (ball_scan.py:267-268, utils.py:1560-1562):
 *   cvdrift_fth = cvdrift + theta0 cvdrift0,  gds2_fth = gds2 + 2 theta0 gds21 + theta0^2 gds22,
 *   g = |gradpar| gds2_fth / bmag,  c = -dPdrho cvdrift_fth / (|gradpar| bmag),
 *   f = gds2_fth / (bmag^3 |gradpar|).
 *   base [nline][8][N], dPdrho [nline], theta0 [nsolve];
 *   line_of_solve [nsolve] or NULL (then line = solve / nth0, i.e. theta0 fastest).
 *   g_out, c_out, f_out [nsolve][N] or NULL: the coefficient arrays gamma_ball_full returns.      */
int ibs_solve_base_batch(const double* base, const double* dPdrho, const double* theta0,
                         const int* line_of_solve, int nth0, int nsolve, int N, double h,
                         const double* lam0, const double* sigma, int chain_len,
                         double* lam_out, double* lam_matrix_out, double* X_out, double* dX_out,
                         double* g_out, double* c_out, double* f_out, int* info_out, void* stream);

/* ---- K4: adjoint (Hellmann-Feynman) gradient -----------------------------------------------------
 * d(lam)/dp = [ int c_p X^2 - int g_p dX^2 - lam int f_p X^2 ] / int f X^2 (utils.py:1666-1680,
 * 1716-1725) for nparam perturbation triples per solve.
 *   lam [nsolve]; X, dX, f [nsolve][N]; g_p, c_p, f_p [nsolve][nparam][N]; grad_out [nsolve][nparam] */
int ibs_adjoint_batch(const double* lam, const double* X, const double* dX, const double* f,
                      const double* g_p, const double* c_p, const double* f_p,
                      int nsolve, int nparam, int N, double* grad_out, void* stream);

/* Per-point sensitivities of lam to the coefficient arrays (what a chained adjoint consumes):
 *   dlam/dg_j = -w_j dX_j^2 / Y1,  dlam/dc_j = w_j X_j^2 / Y1,  dlam/df_j = -lam w_j X_j^2 / Y1,
 * w = Simpson weights, Y1 = int f X^2.  Outputs [nsolve][N] each (any may be NULL).              */
int ibs_adjoint_sensitivities(const double* lam, const double* X, const double* dX, const double* f,
                              int nsolve, int N, double* dlam_dg, double* dlam_dc, double* dlam_df,
                              void* stream);

/* Batched obj_w_grad (utils.py:1632-1728).  For each of npoint (alpha, theta0) points the caller
 * supplies the base arrays of the three field lines alpha-del/2, alpha, alpha+del/2
 * (base3 [npoint][3][8][N], dPdrho3 [npoint][3]); the centre line is solved, d/dtheta0 is analytic
 * (utils.py:1669-1680) and d/dalpha is the central difference of (g, c, f) (utils.py:1707-1725).
 *   val_out [npoint] = -lam; grad_out [npoint][2] = (-dlam/dalpha, -dlam/dtheta0) (utils.py:1728);
 *   lam0 [npoint] or NULL; X_out, dX_out [npoint][N] or NULL; info_out [npoint] or NULL.          */
int ibs_obj_w_grad_batch(const double* base3, const double* dPdrho3, const double* theta0,
                         int npoint, int N, double h, double del_alpha, const double* lam0,
                         double* val_out, double* grad_out, double* X_out, double* dX_out,
                         int* info_out, void* stream);

/* obj_w_grad with the exact alpha-derivative: one field line per point (base [npoint][8][N], dPdrho [npoint]) and its
 * alpha-tangent from ibs_geometry_tangent_batch (dbase [npoint][8][N], ddPdrho [npoint]) instead of three lines.  The
 * solve, val_out, grad_out[:, 1], X_out, dX_out and info_out are those of ibs_obj_w_grad_batch on the same centre lines
 * bit for bit; grad_out[:, 0] = -dlam/dalpha from the chain rule through g, c, f (utils.py:1560-1562) instead of their
 * central difference (utils.py:1707-1725).  lam0 [npoint] or NULL; X_out, dX_out [npoint][N] or NULL; info_out or NULL. */
int ibs_obj_w_grad_tangent_batch(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho,
                                 const double* theta0, int npoint, int N, double h, const double* lam0,
                                 double* val_out, double* grad_out, double* X_out, double* dX_out,
                                 int* info_out, void* stream);

/* ---- scan: per-surface arg-max with the reference's guards (ball_scan.py:279-295) ----------------
 * gamma [ns][ngrid] (row-major (alpha, theta0) grid flattened).  For each surface:
 * max == 0.0 -> idx = -1 (alpha_guess = theta0_guess = 0, sigma0 = 0.05); otherwise the FIRST flat
 * index attaining the maximum (np.where(...)[k][0]); sigma0 = 1.3 |max| + 0.05.
 *   val_out [ns], idx_out [ns], sigma0_out [ns] or NULL                                            */
int ibs_scan_argmax(const double* gamma, int ns, int ngrid, double* val_out, int* idx_out,
                    double* sigma0_out, void* stream);

/* The coarse scan of ball_scan.py:248-295 in ONE call: K2+K3 for nline field lines x nth0 theta0 (theta0 fastest;
 * theta0 [nline*nth0]) with the guarded per-surface arg-max fused into the solver kernel's epilogue (no separate
 * launch): lines_per_surface consecutive field lines form one surface.
 *   best_out [nline/lines_per_surface][2]: packed (max, flat (line-in-surface, theta0) index as a double; -1 = the
 *          all-zero guard, -2 = NaN) -- laid out so that it can BE the send slot of the one all-gather that replaces
 *          the three MPI.Gather of ball_scan.py:345-347;  sigma0_out [nsurf] or NULL;
 *   lam_out [nline*nth0]; X_out, dX_out [nline*nth0][N] or NULL; info_out or NULL; sigma, chain_len as above.       */
int ibs_scan_solve_argmax(const double* base, const double* dPdrho, const double* theta0, int nth0, int nline,
                          int lines_per_surface, int N, double h, const double* sigma, int chain_len,
                          double* lam_out, double* X_out, double* dX_out, int* info_out,
                          double* best_out, double* sigma0_out, void* stream);

/* ---- refinement of the coarse maxima (ball_scan.py:305-314) ---------------------------------------
 * Batched, device-resident replacement of the per-surface scipy L-BFGS-B call
 *   minimize(obj_w_grad, x0=(alpha_guess, theta0_guess), jac=True, bounds=((0, pi), (0, pi/2)),
 *            options={"ftol": 5e-11, "gtol": 2e-8, "maxiter": 30}):
 * a projected quasi-Newton method that advances n problems in lock step.  One round = ibs_geometry_batch on
 * alphas3 (three field lines per problem, alpha_per_surface = 1) -> ibs_obj_w_grad_batch at theta0 -> ibs_refine_step,
 * which consumes (val, grad, info), updates every problem and writes the NEXT trial points into alphas3 / theta0.
 *   state [n][ibs_refine_state_doubles()]: opaque per-problem state; doubles 0..1 = current best (alpha, theta0),
 *          2 = F = -lambda there, 18 = status (2 = finished), 19 = reason (1 pgtol, 2 ftol, 3 maxiter, 4 step, 5 failed),
 *          20 = iterations, 21 = function evaluations;
 *   alphas3_out [n][3] = (a - del/2, a, a + del/2) (utils.py:1641-1646); theta0_out [n];
 *   nactive_out (device int, or NULL): number of problems still running after this step.                        */
int ibs_refine_state_doubles(void);
int ibs_refine_init(double* state, int n, const double* alpha0, const double* theta0_0, double alpha_lo, double alpha_hi,
                    double theta0_lo, double theta0_hi, double del_alpha, double* alphas3_out, double* theta0_out,
                    void* stream);
int ibs_refine_step(double* state, int n, const double* val, const double* grad, const int* info, double ftol,
                    double gtol, int maxiter, double del_alpha, double* alphas3_out, double* theta0_out,
                    int* nactive_out, void* stream);

/* ---- marginal-stability classifier ---------------------------------------------------------------
 * Sturm/Newcomb node count of the discretised ballooning operator at a given lam (the s-alpha test
 * of the reference shoots at lam = 0, tests/shifted-circle-s-alpha/bishop_ball_s-alpha.py:90-115):
 * count_out[i] = number of eigenvalues of the pencil greater than lam[i]; unstable <=> count(0) > 0. */
int ibs_count_above_batch(const double* g, const double* c, const double* f, int nsolve, int N, double h,
                          const double* lam, int* count_out, void* stream);

/* ---- end-to-end host entry point -----------------------------------------------------------------
 * Coarse scan of ball_scan.py:248-295 for ns surfaces with HOST buffers: copies the tables to the
 * device, runs K1 (ns x nalpha lines) and K2+K3 with the fused arg-max (ns x nalpha x nth0 solves), and
 * copies gamma [ns][nalpha][nth0], the per-surface (val, idx, sigma0) and the eigenfunctions back:
 *   xbest_out [ns][nl] or NULL: X of each surface's arg-max solve (what ball_scan.py keeps, :322-339);
 *   xall_out  [ns][nalpha][nth0][nl] or NULL: X of EVERY solve (8 nl bytes per solve over PCIe).
 * Synchronous; uploads, kernels and downloads of consecutive chunks of surfaces overlap.            */
int ibs_scan_host(const double* tab_mn, const double* tab_nyq, const double* scal,
                  const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                  int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                  const double* alpha, int nalpha, const double* theta0, int nth0,
                  const double* theta, int nl, double h,
                  double* gamma_out, double* val_out, int* idx_out, double* sigma0_out, double* xbest_out,
                  double* xall_out, int* nbad_out);

#ifdef __cplusplus
}
#endif
#endif /* IBS_B200_H */
