// C ABI of the library (see include/ibs_b200.h).  Thin argument checking + dispatch; no torch types.
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "ibs_common.cuh"
#include "ibs_refine_core.cuh"

namespace ibs {

// ---- defined in the kernel translation units -------------------------------------------------------
int solve_dispatch(const SolveParams& p, bool base, bool count_only, cudaStream_t stream);
int geometry_dispatch(const double* tab_mn, const double* tab_nyq, const double* scal,
                      const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                      int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                      const double* alpha, int nalpha, int alpha_per_surface, const double* theta, int nl,
                      double phi_center, double* base_out, double* dPdrho_out, double* theta_vmec_out,
                      int* info_out, cudaStream_t st);
int geometry_tangent_dispatch(const double* tab_mn, const double* tab_nyq, const double* scal,
                              const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                              int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                              const double* alpha, int nalpha, int alpha_per_surface, const double* theta, int nl,
                              double phi_center, double* base_out, double* dPdrho_out, double* dbase_out, double* ddPdrho_out,
                              double* theta_vmec_out, int* info_out, cudaStream_t st);
int launch_obj_grad_tangent(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho, const double* theta0,
                            const double* lam, const double* X, const double* dX, int npoint, int N, double* val, double* grad,
                            cudaStream_t st);
int launch_identity_lines(int* line, int n, cudaStream_t st);
int marginal_dispatch(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve, int nth0, int nsolve,
                      int N, double h, double kappa_max, double rtol, double* kappa_out, double* dlam_dkappa_out,
                      double* dkappa_dtheta0_out, double* X_out, int* info_out, cudaStream_t st);
int marginal_tangent_dispatch(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho, const double* theta0,
                              const int* line_of_solve, int nth0, int nsolve, int N, double h, double kappa_max, double rtol,
                              double* kappa_out, double* grad_out, double* X_out, int* info_out, cudaStream_t st);
int marginal_sensitivity_dispatch(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve, int nth0,
                                  int nsolve, int N, double h, const double* kappa, const double* X, double* dk_dg, double* dk_dc,
                                  cudaStream_t st);
int launch_adjoint(const double* lam, const double* X, const double* dX, const double* f, const double* g_p,
                   const double* c_p, const double* f_p, int nsolve, int nparam, int N, double* grad, cudaStream_t st);
int launch_sensitivity(const double* lam, const double* X, const double* dX, const double* f, int nsolve, int N,
                       double* dg, double* dc, double* df, cudaStream_t st);
int launch_obj_grad(const double* base3, const double* dPdrho3, const double* theta0, const double* lam,
                    const double* X, const double* dX, int npoint, int N, double del_alpha, double* val,
                    double* grad, cudaStream_t st);
int launch_centre_lines(int* line, int n, cudaStream_t st);
int launch_argmax(const double* gamma, int ns, int ngrid, double* val, int* idx, double* sigma0, cudaStream_t st);
int launch_argmax_packed(const double* gamma, int ns, int ngrid, double* best, double* sigma0, cudaStream_t st);
bool scan_solver_eligible(const SolveParams& p);
int geometry_adjoint_dispatch(const double* tab_mn, const double* tab_nyq, const double* scal, const double* xm, const double* xn,
                              const double* xm_nyq, const double* xn_nyq, int ns, int mnmax, int mnmax_nyq, double phiedge,
                              double aminor_p, const double* alpha, const double* theta, int nl, double phi_center,
                              const double* theta0, const double* dPdrho, const double* sg, const double* sc, const double* sf,
                              const double* Q, double* grad_mn, double* grad_nyq, double* grad_scal, double* grad_glob,
                              cudaStream_t st);
int geometry_full_nfields();
int geometry_full_dispatch(const double* tab_mn, const double* tab_nyq, const double* bsupumnc, const double* scal,
                           const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                           int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p, const double* alpha, int nalpha,
                           const double* grid, int nl, int mode, double theta_shift, int zero_xn_nyq, double phi_center,
                           double* out, int* info, cudaStream_t st);
int launch_refine_init(double* state, int n, const double* a0, const double* t0, double alo, double ahi, double tlo, double thi,
                       double del_alpha, double* alphas3, double* theta0, cudaStream_t st);
int launch_refine_step(double* state, int n, const double* val, const double* grad, const int* info, double ftol, double gtol,
                       int maxiter, double del_alpha, double* alphas3, double* theta0, int* nactive, cudaStream_t st);
int launch_gather_best(const double* X, const int* idx, int ns, int ngrid, int N, double* out, cudaStream_t st);
int launch_best_setup(const double* best, const double* theta0, int ns, int ngrid, int nth0, double* val_out, int* idx_out,
                      int* line_out, double* th0_out, cudaStream_t st);

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
    return IBS_ERR_CUDA;
}
int num_sms() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (!cached[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

int current_device_slot() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) dev = 0;
    return dev < IBS_MAX_DEVICES ? dev : IBS_MAX_DEVICES - 1;
}

// Warm-start chain used by the scan entry points: consecutive theta0 of one field line (the reference chains
// its ARPACK start vector through the same loop, ball_scan.py:265-274).  The run length divides nth0.
static int scan_chain_len(int nth0) {
    int k = nth0 < 16 ? nth0 : 16;
    while (k > 1 && nth0 % k) --k;
    return k;
}

void keep_pool_cached() {
    static bool done[64] = {false};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return;
    cudaMemPool_t pool;
    unsigned long long thr = ~0ULL;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    if (cudaDeviceGetMemPool(&pool, dev) == cudaSuccess) cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);   // (the current pool, should a host framework have replaced the default one)
    done[dev] = true;
}

// theta0 of every solve of a scan (theta0 fastest): t0[i] = theta0[i % nth0]
__global__ void replicate_theta0_kernel(const double* __restrict__ theta0, int nth0, long long n, double* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = theta0[i % nth0];
}
// number of solves flagged not-converged / bad-input
__global__ void count_bad_kernel(const int* __restrict__ info, long long n, int* __restrict__ count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool bad = i < n && ((info[i] >> 16) & (IBS_FLAG_NOT_CONVERGED | IBS_FLAG_BAD_INPUT));
    const unsigned m = __ballot_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(count, __popc(m));
}

// Streams and events of ibs_scan_host, created once per device and reused by every call.
constexpr int MAX_HOST_CHUNKS = 8, MAX_HOST_SUBCHUNKS = 8;
struct HostCtx {
    std::mutex mu;
    cudaStream_t st_h = nullptr, st = nullptr, st_d = nullptr;
    std::vector<cudaEvent_t> ev_h, ev_c;
    cudaEvent_t ev_alloc = nullptr, ev_done = nullptr;
    int ensure(int nchunk) {
        if (!st_h) IBS_CUDA_CHECK(cudaStreamCreateWithFlags(&st_h, cudaStreamNonBlocking));
        if (!st) IBS_CUDA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        if (!st_d) IBS_CUDA_CHECK(cudaStreamCreateWithFlags(&st_d, cudaStreamNonBlocking));
        if (!ev_alloc) IBS_CUDA_CHECK(cudaEventCreateWithFlags(&ev_alloc, cudaEventDisableTiming));
        if (!ev_done) IBS_CUDA_CHECK(cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming));
        while ((int)ev_h.size() < nchunk) { cudaEvent_t e; IBS_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ev_h.push_back(e); }
        while ((int)ev_c.size() < nchunk) { cudaEvent_t e; IBS_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); ev_c.push_back(e); }
        return IBS_OK;
    }
};
static HostCtx& host_ctx() {
    static HostCtx ctx[IBS_MAX_DEVICES];
    return ctx[current_device_slot()];
}

// FP64 peak probe: independent DFMA chains, 8 per thread, 32 warps per SM (the denominator of the FP64-pipe rooflines)
constexpr int PROBE_CHAINS = 8, PROBE_UNROLL = 16, PROBE_THREADS = 256, PROBE_CTAS_PER_SM = 4;
__global__ void __launch_bounds__(PROBE_THREADS) fp64_probe_kernel(double* __restrict__ out, int iters, double a, double b) {
    double x[PROBE_CHAINS];
#pragma unroll
    for (int c = 0; c < PROBE_CHAINS; ++c) x[c] = 1e-3 * threadIdx.x + c;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < PROBE_UNROLL; ++u)
#pragma unroll
            for (int c = 0; c < PROBE_CHAINS; ++c) x[c] = fma(x[c], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < PROBE_CHAINS; ++c) s += x[c];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

static SolveParams blank_params() { SolveParams p; std::memset(&p, 0, sizeof(p)); return p; }

}  // namespace ibs

using namespace ibs;

extern "C" {

int ibs_version(void) { return 100; }
const char* ibs_last_error(void) { return g_err.c_str(); }

int ibs_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    IBS_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    IBS_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return IBS_OK;
}

int ibs_fp64_probe(int iters, double* scratch, long long scratch_len, double* fma_count_out, void* stream) {
    IBS_REQUIRE(iters >= 1 && scratch && fma_count_out, "bad arguments");
    const int grid = num_sms() * PROBE_CTAS_PER_SM;
    IBS_REQUIRE(scratch_len >= (long long)grid * PROBE_THREADS, "scratch too small (need 4 * SMs * 256 doubles)");
    fp64_probe_kernel<<<grid, PROBE_THREADS, 0, (cudaStream_t)stream>>>(scratch, iters, 0.999, 1e-3);
    IBS_CUDA_CHECK(cudaGetLastError());
    *fma_count_out = (double)grid * PROBE_THREADS * (double)iters * PROBE_UNROLL * PROBE_CHAINS;
    return IBS_OK;
}

int ibs_geometry_batch(const double* tab_mn, const double* tab_nyq, const double* scal,
                       const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                       int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                       const double* alpha, int nalpha, int alpha_per_surface,
                       const double* theta, int nl, double phi_center,
                       double* base_out, double* dPdrho_out, double* theta_vmec_out, int* info_out, void* stream) {
    IBS_REQUIRE(tab_mn && tab_nyq && scal && xm && xn && xm_nyq && xn_nyq && alpha && theta && base_out, "null pointer");
    IBS_REQUIRE(ns >= 0 && nalpha >= 0 && nl >= 1 && mnmax >= 1 && mnmax_nyq >= 1, "bad sizes");
    IBS_REQUIRE(aminor_p > 0.0 && phiedge != 0.0, "Aminor_p must be > 0 and phiedge != 0");
    if (ns == 0 || nalpha == 0) return IBS_OK;
    return geometry_dispatch(tab_mn, tab_nyq, scal, xm, xn, xm_nyq, xn_nyq, ns, mnmax, mnmax_nyq, phiedge, aminor_p, alpha,
                             nalpha, alpha_per_surface, theta, nl, phi_center, base_out, dPdrho_out, theta_vmec_out,
                             info_out, (cudaStream_t)stream);
}

int ibs_geometry_tangent_batch(const double* tab_mn, const double* tab_nyq, const double* scal,
                               const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                               int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                               const double* alpha, int nalpha, int alpha_per_surface,
                               const double* theta, int nl, double phi_center, double* base_out, double* dPdrho_out,
                               double* dbase_out, double* ddPdrho_out, double* theta_vmec_out, int* info_out, void* stream) {
    IBS_REQUIRE(tab_mn && tab_nyq && scal && xm && xn && xm_nyq && xn_nyq && alpha && theta && base_out && dbase_out, "null pointer");
    IBS_REQUIRE(ns >= 0 && nalpha >= 0 && nl >= 1 && mnmax >= 1 && mnmax_nyq >= 1, "bad sizes");
    IBS_REQUIRE(aminor_p > 0.0 && phiedge != 0.0, "Aminor_p must be > 0 and phiedge != 0");
    if (ns == 0 || nalpha == 0) return IBS_OK;
    return geometry_tangent_dispatch(tab_mn, tab_nyq, scal, xm, xn, xm_nyq, xn_nyq, ns, mnmax, mnmax_nyq, phiedge, aminor_p, alpha,
                                     nalpha, alpha_per_surface, theta, nl, phi_center, base_out, dPdrho_out, dbase_out, ddPdrho_out,
                                     theta_vmec_out, info_out, (cudaStream_t)stream);
}

int ibs_geometry_full_nfields(void) { return geometry_full_nfields(); }

int ibs_geometry_full(const double* tab_mn, const double* tab_nyq, const double* bsupumnc, const double* scal,
                      const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                      int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                      const double* alpha, int nalpha, const double* grid, int nl, int mode, double theta_shift,
                      int zero_xn_nyq, double phi_center, double* out, int* info_out, void* stream) {
    IBS_REQUIRE(tab_mn && tab_nyq && bsupumnc && scal && xm && xn && xm_nyq && xn_nyq && alpha && grid && out, "null pointer");
    IBS_REQUIRE(ns >= 0 && nalpha >= 0 && nl >= 1 && mnmax >= 1 && mnmax_nyq >= 1 && mode >= 0 && mode <= 2, "bad sizes / mode");
    IBS_REQUIRE(aminor_p > 0.0 && phiedge != 0.0, "Aminor_p must be > 0 and phiedge != 0");
    return geometry_full_dispatch(tab_mn, tab_nyq, bsupumnc, scal, xm, xn, xm_nyq, xn_nyq, ns, mnmax, mnmax_nyq, phiedge, aminor_p,
                                  alpha, nalpha, grid, nl, mode, theta_shift, zero_xn_nyq, phi_center, out, info_out,
                                  (cudaStream_t)stream);
}

int ibs_geometry_adjoint(const double* tab_mn, const double* tab_nyq, const double* scal,
                         const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                         int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                         const double* alpha, const double* theta, int nl, double phi_center,
                         const double* theta0, const double* dPdrho, const double* dlam_dg, const double* dlam_dc,
                         const double* dlam_df, const double* Q, double* grad_mn_out, double* grad_nyq_out, void* stream) {
    IBS_REQUIRE(ns >= 0 && nl >= 1 && mnmax >= 1 && mnmax_nyq >= 1, "bad sizes");
    if (ns == 0) return IBS_OK;
    IBS_REQUIRE(tab_mn && tab_nyq && scal && xm && xn && xm_nyq && xn_nyq && alpha && theta && theta0 && dPdrho && dlam_dg && dlam_dc &&
                dlam_df && Q && grad_mn_out && grad_nyq_out, "null pointer");
    IBS_REQUIRE(aminor_p > 0.0 && phiedge != 0.0, "Aminor_p must be > 0 and phiedge != 0");
    return geometry_adjoint_dispatch(tab_mn, tab_nyq, scal, xm, xn, xm_nyq, xn_nyq, ns, mnmax, mnmax_nyq, phiedge, aminor_p, alpha, theta,
                                     nl, phi_center, theta0, dPdrho, dlam_dg, dlam_dc, dlam_df, Q, grad_mn_out, grad_nyq_out, nullptr,
                                     nullptr, (cudaStream_t)stream);
}

int ibs_geometry_adjoint_scal(const double* tab_mn, const double* tab_nyq, const double* scal,
                              const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                              int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                              const double* alpha, const double* theta, int nl, double phi_center,
                              const double* theta0, const double* dPdrho, const double* dlam_dg, const double* dlam_dc,
                              const double* dlam_df, const double* Q, double* grad_mn_out, double* grad_nyq_out,
                              double* grad_scal_out, double* grad_glob_out, void* stream) {
    IBS_REQUIRE(ns >= 0 && nl >= 1 && mnmax >= 1 && mnmax_nyq >= 1, "bad sizes");
    if (ns == 0) return IBS_OK;
    IBS_REQUIRE(tab_mn && tab_nyq && scal && xm && xn && xm_nyq && xn_nyq && alpha && theta && theta0 && dPdrho && dlam_dg && dlam_dc &&
                dlam_df && Q && grad_mn_out && grad_nyq_out && grad_scal_out && grad_glob_out, "null pointer");
    IBS_REQUIRE(aminor_p > 0.0 && phiedge != 0.0, "Aminor_p must be > 0 and phiedge != 0");
    return geometry_adjoint_dispatch(tab_mn, tab_nyq, scal, xm, xn, xm_nyq, xn_nyq, ns, mnmax, mnmax_nyq, phiedge, aminor_p, alpha, theta,
                                     nl, phi_center, theta0, dPdrho, dlam_dg, dlam_dc, dlam_df, Q, grad_mn_out, grad_nyq_out,
                                     grad_scal_out, grad_glob_out, (cudaStream_t)stream);
}

int ibs_solve_gcf_batch(const double* g, const double* c, const double* f, int nsolve, int N, double h,
                        const double* lam0, const double* sigma, int chain_len, double* lam_out, double* lam_matrix_out,
                        double* X_out, double* dX_out, int* info_out, void* stream) {
    IBS_REQUIRE(nsolve >= 0 && N >= 5, "need nsolve >= 0 and N >= 5");
    if (nsolve == 0) return IBS_OK;                 // empty batches are legal (and have null pointers)
    IBS_REQUIRE(g && c && f && lam_out, "null pointer");
    IBS_REQUIRE(h > 0.0, "h must be positive");
    SolveParams p = blank_params();
    p.g = g; p.c = c; p.f = f; p.nsolve = nsolve; p.N = N; p.h = h; p.lam0 = lam0; p.sigma = sigma; p.chain_len = chain_len;
    p.lam_out = lam_out; p.lam_matrix_out = lam_matrix_out; p.X_out = X_out; p.dX_out = dX_out; p.info_out = info_out;
    return solve_dispatch(p, false, false, (cudaStream_t)stream);
}

int ibs_solve_base_batch(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve,
                         int nth0, int nsolve, int N, double h, const double* lam0, const double* sigma, int chain_len,
                         double* lam_out, double* lam_matrix_out, double* X_out, double* dX_out, double* g_out,
                         double* c_out, double* f_out, int* info_out, void* stream) {
    IBS_REQUIRE(nsolve >= 0 && N >= 5, "need nsolve >= 0 and N >= 5");
    if (nsolve == 0) return IBS_OK;
    IBS_REQUIRE(base && dPdrho && theta0 && lam_out, "null pointer");
    IBS_REQUIRE(line_of_solve || nth0 >= 1, "need line_of_solve or nth0 >= 1");
    keep_pool_cached();
    IBS_REQUIRE(h > 0.0, "h must be positive");
    SolveParams p = blank_params();
    p.base = base; p.dPdrho = dPdrho; p.theta0 = theta0; p.line_of_solve = line_of_solve; p.nth0 = nth0 > 0 ? nth0 : 1;
    p.nsolve = nsolve; p.N = N; p.h = h; p.lam0 = lam0; p.sigma = sigma; p.chain_len = chain_len;
    p.lam_out = lam_out; p.lam_matrix_out = lam_matrix_out; p.X_out = X_out; p.dX_out = dX_out;
    p.g_out = g_out; p.c_out = c_out; p.f_out = f_out; p.info_out = info_out;
    return solve_dispatch(p, true, false, (cudaStream_t)stream);
}

int ibs_scan_solve_argmax(const double* base, const double* dPdrho, const double* theta0, int nth0, int nline,
                          int lines_per_surface, int N, double h, const double* sigma, int chain_len,
                          double* lam_out, double* X_out, double* dX_out, int* info_out,
                          double* best_out, double* sigma0_out, void* stream) {
    IBS_REQUIRE(nline >= 0 && nth0 >= 1 && N >= 5 && h > 0.0, "bad sizes");
    IBS_REQUIRE(lines_per_surface >= 1 && nline % lines_per_surface == 0, "nline must be a multiple of lines_per_surface");
    IBS_REQUIRE((long long)nline * nth0 <= 0x7fffffffLL, "nline * nth0 must fit an int");
    if (nline == 0) return IBS_OK;
    IBS_REQUIRE(base && dPdrho && theta0 && lam_out && best_out, "null pointer");
    keep_pool_cached();
    SolveParams p = blank_params();
    p.base = base; p.dPdrho = dPdrho; p.theta0 = theta0; p.nth0 = nth0; p.nsolve = nline * nth0; p.N = N; p.h = h;
    p.sigma = sigma; p.chain_len = chain_len;
    p.lam_out = lam_out; p.X_out = X_out; p.dX_out = dX_out; p.info_out = info_out;
    p.lines_per_surface = lines_per_surface; p.best_out = best_out; p.sigma0_out = sigma0_out;
    cudaStream_t st = (cudaStream_t)stream;
    const bool fused = scan_solver_eligible(p);            // the lane-per-solve kernel reduces in its epilogue
    int rc = solve_dispatch(p, true, false, st);
    if (rc == IBS_OK && !fused)
        rc = launch_argmax_packed(lam_out, nline / lines_per_surface, lines_per_surface * nth0, best_out, sigma0_out, st);
    return rc;
}

int ibs_refine_state_doubles(void) { return ibs::refine::NSTATE; }

int ibs_refine_init(double* state, int n, const double* alpha0, const double* theta0_0, double alpha_lo, double alpha_hi,
                    double theta0_lo, double theta0_hi, double del_alpha, double* alphas3_out, double* theta0_out, void* stream) {
    IBS_REQUIRE(n >= 0 && alpha_lo <= alpha_hi && theta0_lo <= theta0_hi, "bad sizes / bounds");
    if (n == 0) return IBS_OK;
    IBS_REQUIRE(state && alpha0 && theta0_0 && alphas3_out && theta0_out, "null pointer");
    return launch_refine_init(state, n, alpha0, theta0_0, alpha_lo, alpha_hi, theta0_lo, theta0_hi, del_alpha, alphas3_out, theta0_out,
                              (cudaStream_t)stream);
}

int ibs_refine_step(double* state, int n, const double* val, const double* grad, const int* info, double ftol, double gtol,
                    int maxiter, double del_alpha, double* alphas3_out, double* theta0_out, int* nactive_out, void* stream) {
    IBS_REQUIRE(n >= 0 && maxiter >= 1, "bad sizes");
    if (n == 0) return IBS_OK;
    IBS_REQUIRE(state && val && grad && alphas3_out && theta0_out, "null pointer");
    return launch_refine_step(state, n, val, grad, info, ftol, gtol, maxiter, del_alpha, alphas3_out, theta0_out, nactive_out,
                              (cudaStream_t)stream);
}

int ibs_count_above_batch(const double* g, const double* c, const double* f, int nsolve, int N, double h,
                          const double* lam, int* count_out, void* stream) {
    IBS_REQUIRE(nsolve >= 0 && N >= 3 && h > 0.0, "bad sizes");
    if (nsolve == 0) return IBS_OK;
    IBS_REQUIRE(g && c && f && lam && count_out, "null pointer");
    SolveParams p = blank_params();
    p.g = g; p.c = c; p.f = f; p.nsolve = nsolve; p.N = N; p.h = h; p.lam_query = lam; p.count_out = count_out;
    return solve_dispatch(p, false, true, (cudaStream_t)stream);
}

int ibs_marginal_batch(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve,
                       int nth0, int nsolve, int N, double h, double kappa_max, double rtol,
                       double* kappa_out, double* dlam_dkappa_out, double* dkappa_dtheta0_out, double* X_out,
                       int* info_out, void* stream) {
    IBS_REQUIRE(nsolve >= 0 && N >= 5 && N <= 65538, "need nsolve >= 0 and 5 <= N <= 65538");
    if (nsolve == 0) return IBS_OK;
    IBS_REQUIRE(base && dPdrho && theta0 && kappa_out, "null pointer");
    IBS_REQUIRE(line_of_solve || nth0 >= 1, "need line_of_solve or nth0 >= 1");
    IBS_REQUIRE(h > 0.0, "h must be positive");
    IBS_REQUIRE(kappa_max > 0.0 && rtol > 0.0 && rtol < 1.0, "need kappa_max > 0 and 0 < rtol < 1");
    keep_pool_cached();
    return marginal_dispatch(base, dPdrho, theta0, line_of_solve, nth0 > 0 ? nth0 : 1, nsolve, N, h, kappa_max, rtol, kappa_out,
                             dlam_dkappa_out, dkappa_dtheta0_out, X_out, info_out, (cudaStream_t)stream);
}

int ibs_marginal_tangent_batch(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho,
                               const double* theta0, const int* line_of_solve, int nth0, int nsolve, int N, double h,
                               double kappa_max, double rtol, double* kappa_out, double* grad_out, double* X_out, int* info_out,
                               void* stream) {
    IBS_REQUIRE(nsolve >= 0 && N >= 5 && N <= 65538, "need nsolve >= 0 and 5 <= N <= 65538");
    if (nsolve == 0) return IBS_OK;
    IBS_REQUIRE(base && dbase && dPdrho && ddPdrho && theta0 && kappa_out && grad_out, "null pointer");
    IBS_REQUIRE(line_of_solve || nth0 >= 1, "need line_of_solve or nth0 >= 1");
    IBS_REQUIRE(h > 0.0, "h must be positive");
    IBS_REQUIRE(kappa_max > 0.0 && rtol > 0.0 && rtol < 1.0, "need kappa_max > 0 and 0 < rtol < 1");
    keep_pool_cached();
    return marginal_tangent_dispatch(base, dbase, dPdrho, ddPdrho, theta0, line_of_solve, nth0 > 0 ? nth0 : 1, nsolve, N, h, kappa_max,
                                     rtol, kappa_out, grad_out, X_out, info_out, (cudaStream_t)stream);
}

int ibs_marginal_sensitivities(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve, int nth0,
                               int nsolve, int N, double h, const double* kappa, const double* X, double* dkappa_dg_out,
                               double* dkappa_dc_out, void* stream) {
    IBS_REQUIRE(nsolve >= 0 && N >= 5 && N <= 65538, "need nsolve >= 0 and 5 <= N <= 65538");
    if (nsolve == 0) return IBS_OK;
    IBS_REQUIRE(base && dPdrho && theta0 && kappa && X && dkappa_dg_out && dkappa_dc_out, "null pointer");
    IBS_REQUIRE(line_of_solve || nth0 >= 1, "need line_of_solve or nth0 >= 1");
    IBS_REQUIRE(h > 0.0, "h must be positive");
    return marginal_sensitivity_dispatch(base, dPdrho, theta0, line_of_solve, nth0 > 0 ? nth0 : 1, nsolve, N, h, kappa, X,
                                         dkappa_dg_out, dkappa_dc_out, (cudaStream_t)stream);
}

int ibs_adjoint_batch(const double* lam, const double* X, const double* dX, const double* f, const double* g_p,
                      const double* c_p, const double* f_p, int nsolve, int nparam, int N, double* grad_out,
                      void* stream) {
    IBS_REQUIRE(nsolve >= 0 && nparam >= 0 && N >= 3, "bad sizes");
    if (nsolve == 0 || nparam == 0) return IBS_OK;
    IBS_REQUIRE(lam && X && dX && f && g_p && c_p && f_p && grad_out, "null pointer");
    return launch_adjoint(lam, X, dX, f, g_p, c_p, f_p, nsolve, nparam, N, grad_out, (cudaStream_t)stream);
}

int ibs_adjoint_sensitivities(const double* lam, const double* X, const double* dX, const double* f, int nsolve,
                              int N, double* dlam_dg, double* dlam_dc, double* dlam_df, void* stream) {
    IBS_REQUIRE(nsolve >= 0 && N >= 3, "bad sizes");
    if (nsolve == 0) return IBS_OK;
    IBS_REQUIRE(lam && X && dX && f, "null pointer");
    return launch_sensitivity(lam, X, dX, f, nsolve, N, dlam_dg, dlam_dc, dlam_df, (cudaStream_t)stream);
}

int ibs_obj_w_grad_batch(const double* base3, const double* dPdrho3, const double* theta0, int npoint, int N,
                         double h, double del_alpha, const double* lam0, double* val_out, double* grad_out,
                         double* X_out, double* dX_out, int* info_out, void* stream) {
    IBS_REQUIRE(npoint >= 0 && N >= 5 && h > 0.0 && del_alpha != 0.0, "bad sizes");
    if (npoint == 0) return IBS_OK;
    IBS_REQUIRE(base3 && dPdrho3 && theta0 && val_out && grad_out, "null pointer");
    IBS_REQUIRE((long long)npoint * 3 <= 0x7fffffffLL, "npoint too large (3 * npoint field lines must fit an int)");
    cudaStream_t st = (cudaStream_t)stream;
    // stream-ordered scratch: centre-line indices, lambda, and X / dX when the caller does not want them -- ONE
    // allocation, so that no error path can leak a part of it
    const size_t o_line = 0, o_lam = ((size_t)npoint * sizeof(int) + 255) & ~(size_t)255;
    const size_t o_X = o_lam + (((size_t)npoint * sizeof(double) + 255) & ~(size_t)255);
    const size_t xbytes = ((size_t)npoint * N * sizeof(double) + 255) & ~(size_t)255;
    const size_t o_dX = o_X + (X_out ? 0 : xbytes), total = o_dX + (dX_out ? 0 : xbytes);
    char* ws = nullptr;
    IBS_CUDA_CHECK(cudaMallocAsync((void**)&ws, total + 256, st));
    int* line = (int*)(ws + o_line);
    double* lam = (double*)(ws + o_lam);
    double* X = X_out ? X_out : (double*)(ws + o_X);
    double* dX = dX_out ? dX_out : (double*)(ws + o_dX);
    int rc = launch_centre_lines(line, npoint, st);
    if (rc == IBS_OK) {
        SolveParams p = blank_params();
        p.base = base3; p.dPdrho = dPdrho3; p.theta0 = theta0; p.line_of_solve = line; p.nth0 = 1;
        p.nsolve = npoint; p.N = N; p.h = h; p.lam0 = lam0;
        p.lam_out = lam; p.X_out = X; p.dX_out = dX; p.info_out = info_out;
        rc = solve_dispatch(p, true, false, st);
    }
    if (rc == IBS_OK) rc = launch_obj_grad(base3, dPdrho3, theta0, lam, X, dX, npoint, N, del_alpha, val_out, grad_out, st);
    cudaFreeAsync(ws, st);
    return rc;
}

int ibs_obj_w_grad_tangent_batch(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho,
                                 const double* theta0, int npoint, int N, double h, const double* lam0, double* val_out,
                                 double* grad_out, double* X_out, double* dX_out, int* info_out, void* stream) {
    IBS_REQUIRE(npoint >= 0 && N >= 5 && h > 0.0, "bad sizes");
    if (npoint == 0) return IBS_OK;
    IBS_REQUIRE(base && dbase && dPdrho && ddPdrho && theta0 && val_out && grad_out, "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    // the solve is ibs_obj_w_grad_batch's (explicit line per solve, same kernel choice) on line i instead of 3 i + 1
    const size_t o_line = 0, o_lam = ((size_t)npoint * sizeof(int) + 255) & ~(size_t)255;
    const size_t o_X = o_lam + (((size_t)npoint * sizeof(double) + 255) & ~(size_t)255);
    const size_t xbytes = ((size_t)npoint * N * sizeof(double) + 255) & ~(size_t)255;
    const size_t o_dX = o_X + (X_out ? 0 : xbytes), total = o_dX + (dX_out ? 0 : xbytes);
    char* ws = nullptr;
    IBS_CUDA_CHECK(cudaMallocAsync((void**)&ws, total + 256, st));
    int* line = (int*)(ws + o_line);
    double* lam = (double*)(ws + o_lam);
    double* X = X_out ? X_out : (double*)(ws + o_X);
    double* dX = dX_out ? dX_out : (double*)(ws + o_dX);
    int rc = launch_identity_lines(line, npoint, st);
    if (rc == IBS_OK) {
        SolveParams p = blank_params();
        p.base = base; p.dPdrho = dPdrho; p.theta0 = theta0; p.line_of_solve = line; p.nth0 = 1;
        p.nsolve = npoint; p.N = N; p.h = h; p.lam0 = lam0;
        p.lam_out = lam; p.X_out = X; p.dX_out = dX; p.info_out = info_out;
        rc = solve_dispatch(p, true, false, st);
    }
    if (rc == IBS_OK) rc = launch_obj_grad_tangent(base, dbase, dPdrho, ddPdrho, theta0, lam, X, dX, npoint, N, val_out, grad_out, st);
    cudaFreeAsync(ws, st);
    return rc;
}

int ibs_scan_argmax(const double* gamma, int ns, int ngrid, double* val_out, int* idx_out, double* sigma0_out,
                    void* stream) {
    IBS_REQUIRE(gamma && val_out && idx_out, "null pointer");
    IBS_REQUIRE(ns >= 0 && ngrid >= 1, "bad sizes");
    return launch_argmax(gamma, ns, ngrid, val_out, idx_out, sigma0_out, (cudaStream_t)stream);
}

int ibs_scan_host(const double* tab_mn, const double* tab_nyq, const double* scal,
                  const double* xm, const double* xn, const double* xm_nyq, const double* xn_nyq,
                  int ns, int mnmax, int mnmax_nyq, double phiedge, double aminor_p,
                  const double* alpha, int nalpha, const double* theta0, int nth0,
                  const double* theta, int nl, double h,
                  double* gamma_out, double* val_out, int* idx_out, double* sigma0_out, double* xbest_out, double* xall_out,
                  int* nbad_out) {
    IBS_REQUIRE(tab_mn && tab_nyq && scal && alpha && theta0 && theta && gamma_out, "null pointer");
    IBS_REQUIRE(ns >= 1 && nalpha >= 1 && nth0 >= 1 && nl >= 3, "bad sizes");
    IBS_REQUIRE((long long)ns * nalpha * nth0 <= 0x7fffffffLL, "ns * nalpha * nth0 must fit an int");
    keep_pool_cached();
    // Three streams: uploads, compute, downloads.  The surfaces are processed in chunks (every chunk: tables up ->
    // K1 -> K2+K3 -> arg-max -> eigenfunction of each surface's maximum -> results down), so that the copies of one chunk
    // overlap the kernels of its neighbours (chunk boundaries cb[] below).
    // Streams and events are created once per device and reused (the call holds the device's context lock).
    HostCtx& hc = host_ctx();
    std::lock_guard<std::mutex> hold(hc.mu);
    if (int rc0 = hc.ensure(MAX_HOST_CHUNKS * (MAX_HOST_SUBCHUNKS + 1))) return rc0;
    cudaStream_t st_h = hc.st_h, st = hc.st, st_d = hc.st_d;
    const size_t nlines = (size_t)ns * nalpha, nsolve = nlines * nth0;
    const int ngrid = nalpha * nth0;
    // Chunks of >= 8 rounds of the lane kernel's resident warps (ONE solver launch per chunk: the lane kernel warm-starts
    // every line after its first two rounds, so short launches are slow launches), each cut into NSUB sub-chunks for the
    // copies: tables of sub-chunk i+1 go up while K1 runs on sub-chunk i, the eigenfunctions of sub-chunk i go down while
    // those of i+1 are re-solved.  Only 1/NSUB of the first upload and of the last download overlap nothing.
    // Measured, D3D config x 37 equilibria (solves/s): equal chunks with their own solver launch 1 / 2 / 3 / 4 / 6 =
    // 5.3e7 / 6.4e7 / 5.6e7 / 5.5e7 / 5.0e7; small first / last chunks 6.0e7; this form with 1 / 2 / 4 / 8 sub-chunks:
    // 6.1e7 / 6.9e7 / 7.2e7 / 7.1e7.
    // IBS_HOST_CHUNKS / IBS_HOST_SUBCHUNKS override.
    std::vector<size_t> cb;
    int nsub = 4;
    {
        const int grp = (nth0 + 15) / 16;
        const long long items = (long long)nlines * grp, per_round = 16LL * num_sms();
        int n = (int)(items / (8 * per_round));
        if (const char* e = std::getenv("IBS_HOST_CHUNKS")) n = std::atoi(e);
        if (n > MAX_HOST_CHUNKS) n = MAX_HOST_CHUNKS;
        if (n > ns) n = ns;
        if (n < 1) n = 1;
        for (int c = 0; c <= n; ++c) cb.push_back((size_t)ns * c / n);
        {   // sub-chunks pay only when a chunk's copies are large (>= 4 MB each); small ones cost K1 its full-size launches
            const size_t per_surface = (size_t)(6 * mnmax + 7 * mnmax_nyq + IBS_NSCAL) * 8;
            const size_t up = per_surface * (size_t)ns / n, down = xbest_out ? (size_t)nl * 8 * (size_t)ns / n : 0;
            const size_t big = up > down ? up : down;
            nsub = (int)(big / ((size_t)4 << 20));
            if (nsub > 4) nsub = 4;
        }
        if (const char* e = std::getenv("IBS_HOST_SUBCHUNKS")) nsub = std::atoi(e);
        if (nsub > MAX_HOST_SUBCHUNKS) nsub = MAX_HOST_SUBCHUNKS;
        if ((size_t)nsub > (size_t)ns / n) nsub = (int)((size_t)ns / n);
        if (nsub < 1) nsub = 1;
    }
    const int nchunk = (int)cb.size() - 1;
    auto sub_lo = [&](int c, int q) { return cb[c] + (cb[c + 1] - cb[c]) * (size_t)q / (size_t)nsub; };      // first surface of sub-chunk q of chunk c
    const size_t r_mn = (size_t)6 * mnmax * 8, r_nyq = (size_t)7 * mnmax_nyq * 8, r_sc = (size_t)IBS_NSCAL * 8;      // bytes per surface
    // one device arena: inputs | base | dPdrho | theta0 per solve | gamma | val | sigma0 | idx | info | best-solve scratch
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_tmn = take(ns * r_mn), o_tnq = take(ns * r_nyq), o_sc = take(ns * r_sc), o_al = take((size_t)nalpha * 8),
                 o_th = take((size_t)nl * 8), o_t0 = take(nsolve * 8), o_base = take(nlines * IBS_NBASE * nl * 8),
                 o_dp = take(nlines * 8), o_gam = take(nsolve * 8), o_val = take((size_t)ns * 8), o_sig = take((size_t)ns * 8),
                 o_idx = take((size_t)ns * 4), o_info = take(nsolve * 4),
                 o_xb = take(xbest_out ? (size_t)ns * nl * 8 : 0), o_bl = take((size_t)ns * 4), o_bt = take((size_t)ns * 8),
                 o_bg = take((size_t)ns * 8), o_t0h = take((size_t)nth0 * 8), o_nb = take(4), o_best = take((size_t)ns * 16),
                 o_xa = take(xall_out ? nsolve * nl * 8 : 0);
    char* d = nullptr;
    int rc = IBS_OK;
    int nbad_host = 0;
    std::vector<cudaEvent_t>& ev_h = hc.ev_h; std::vector<cudaEvent_t>& ev_c = hc.ev_c;
    cudaEvent_t ev_alloc = hc.ev_alloc, ev_done = hc.ev_done;
#define IBS_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { rc = cuda_fail(_e, #expr); goto done; } } while (0)
    IBS_TRY(cudaMallocAsync((void**)&d, off, st));
    IBS_TRY(cudaEventRecord(ev_alloc, st));
    IBS_TRY(cudaStreamWaitEvent(st_h, ev_alloc, 0));
    IBS_TRY(cudaStreamWaitEvent(st_d, ev_alloc, 0));
    // ---- uploads: the small arrays first, then the tables chunk by chunk
    IBS_TRY(cudaMemcpyAsync(d + o_al, alpha, (size_t)nalpha * 8, cudaMemcpyHostToDevice, st_h));
    IBS_TRY(cudaMemcpyAsync(d + o_th, theta, (size_t)nl * 8, cudaMemcpyHostToDevice, st_h));
    IBS_TRY(cudaMemcpyAsync(d + o_t0h, theta0, (size_t)nth0 * 8, cudaMemcpyHostToDevice, st_h));
    replicate_theta0_kernel<<<(unsigned)((nsolve + 255) / 256), 256, 0, st_h>>>((double*)(d + o_t0h), nth0, (long long)nsolve, (double*)(d + o_t0));
    IBS_TRY(cudaGetLastError());
    IBS_TRY(cudaMemsetAsync(d + o_nb, 0, 4, st_h));
    for (int c = 0; c < nchunk; ++c)
        for (int q = 0; q < nsub; ++q) {
            const size_t s0 = sub_lo(c, q), nsc = sub_lo(c, q + 1) - s0;
            IBS_TRY(cudaMemcpyAsync(d + o_tmn + s0 * r_mn, (const char*)tab_mn + s0 * r_mn, nsc * r_mn, cudaMemcpyHostToDevice, st_h));
            IBS_TRY(cudaMemcpyAsync(d + o_tnq + s0 * r_nyq, (const char*)tab_nyq + s0 * r_nyq, nsc * r_nyq, cudaMemcpyHostToDevice, st_h));
            IBS_TRY(cudaMemcpyAsync(d + o_sc + s0 * r_sc, (const char*)scal + s0 * r_sc, nsc * r_sc, cudaMemcpyHostToDevice, st_h));
            IBS_TRY(cudaEventRecord(ev_h[c * nsub + q], st_h));
        }
    // ---- compute + downloads, chunk by chunk
    for (int c = 0; c < nchunk; ++c) {
        const size_t s0 = cb[c], nsc = cb[c + 1] - s0;
        const size_t l0 = s0 * nalpha, nlc = nsc * nalpha, v0 = l0 * nth0, nvc = nlc * nth0;
        double* base_c = (double*)(d + o_base) + l0 * IBS_NBASE * nl;
        double* dp_c = (double*)(d + o_dp) + l0;
        // K1, sub-chunk by sub-chunk as the tables arrive
        for (int q = 0; q < nsub; ++q) {
            const size_t q0 = sub_lo(c, q), nq = sub_lo(c, q + 1) - q0;
            IBS_TRY(cudaStreamWaitEvent(st, ev_h[c * nsub + q], 0));
            rc = geometry_dispatch((double*)(d + o_tmn + q0 * r_mn), (double*)(d + o_tnq + q0 * r_nyq), (double*)(d + o_sc + q0 * r_sc), xm, xn,
                                   xm_nyq, xn_nyq, (int)nq, mnmax, mnmax_nyq, phiedge, aminor_p, (double*)(d + o_al), nalpha, 0,
                                   (double*)(d + o_th), nl, 0.0, (double*)(d + o_base) + q0 * nalpha * IBS_NBASE * nl,
                                   (double*)(d + o_dp) + q0 * nalpha, nullptr, nullptr, st);
            if (rc != IBS_OK) goto done;
        }
        {
            // K2+K3 with the per-surface arg-max fused into the solver's epilogue (one packed (max, index) pair per surface)
            SolveParams p = blank_params();
            p.base = base_c; p.dPdrho = dp_c; p.theta0 = (double*)(d + o_t0) + v0; p.nth0 = nth0;
            p.nsolve = (int)nvc; p.N = nl; p.h = h; p.lam_out = (double*)(d + o_gam) + v0; p.info_out = (int*)(d + o_info) + v0;
            p.X_out = xall_out ? (double*)(d + o_xa) + v0 * nl : nullptr;
            p.chain_len = scan_chain_len(nth0);
            p.lines_per_surface = nalpha; p.best_out = (double*)(d + o_best) + 2 * s0; p.sigma0_out = (double*)(d + o_sig) + s0;
            const bool fused = scan_solver_eligible(p);
            rc = solve_dispatch(p, true, false, st);
            if (rc == IBS_OK && !fused) rc = launch_argmax_packed(p.lam_out, (int)nsc, ngrid, p.best_out, p.sigma0_out, st);
            if (rc != IBS_OK) goto done;
        }
        // val / idx for the host and the (line, theta0) of each surface's maximum; line indices are chunk-local
        rc = launch_best_setup((double*)(d + o_best) + 2 * s0, (double*)(d + o_t0) + v0, (int)nsc, ngrid, nth0, (double*)(d + o_val) + s0,
                               (int*)(d + o_idx) + s0, (int*)(d + o_bl) + s0, (double*)(d + o_bt) + s0, st);
        if (rc != IBS_OK) goto done;
        count_bad_kernel<<<(unsigned)((nvc + 255) / 256), 256, 0, st>>>((int*)(d + o_info) + v0, (long long)nvc, (int*)(d + o_nb));
        IBS_TRY(cudaGetLastError());
        // the grid results go down while the eigenfunctions are formed
        IBS_TRY(cudaEventRecord(ev_c[c * (nsub + 1)], st));
        IBS_TRY(cudaStreamWaitEvent(st_d, ev_c[c * (nsub + 1)], 0));
        IBS_TRY(cudaMemcpyAsync(gamma_out + v0, d + o_gam + v0 * 8, nvc * 8, cudaMemcpyDeviceToHost, st_d));
        if (val_out) IBS_TRY(cudaMemcpyAsync(val_out + s0, d + o_val + s0 * 8, nsc * 8, cudaMemcpyDeviceToHost, st_d));
        if (idx_out) IBS_TRY(cudaMemcpyAsync(idx_out + s0, d + o_idx + s0 * 4, nsc * 4, cudaMemcpyDeviceToHost, st_d));
        if (sigma0_out) IBS_TRY(cudaMemcpyAsync(sigma0_out + s0, d + o_sig + s0 * 8, nsc * 8, cudaMemcpyDeviceToHost, st_d));
        for (int q = 0; q < nsub && (xbest_out || xall_out); ++q) {
            const size_t q0 = sub_lo(c, q), nq = sub_lo(c, q + 1) - q0;
            const size_t qv0 = q0 * nalpha * nth0, nqv = nq * nalpha * nth0;
            if (xbest_out && !xall_out) {
                // eigenfunction of each surface's arg-max only: re-solve those problems with the eigenvector written out
                // (instead of writing nsolve eigenvectors and gathering ns of them); line indices are chunk-local
                SolveParams pb = blank_params();
                pb.base = base_c; pb.dPdrho = dp_c; pb.theta0 = (double*)(d + o_bt) + q0;
                pb.line_of_solve = (int*)(d + o_bl) + q0; pb.nth0 = 1; pb.nsolve = (int)nq; pb.N = nl; pb.h = h;
                pb.lam_out = (double*)(d + o_bg) + q0; pb.X_out = (double*)(d + o_xb) + q0 * nl;
                pb.lam0 = (double*)(d + o_val) + q0;          // warm start: the maximum itself (a NaN / guarded entry fails the bracket test: cold start)
                rc = solve_dispatch(pb, true, false, st);
                if (rc != IBS_OK) goto done;
            } else if (xbest_out) {
                // idx is local to the surface; the gather kernel takes this sub-chunk's first solve as its base
                rc = launch_gather_best((double*)(d + o_xa) + qv0 * nl, (int*)(d + o_idx) + q0, (int)nq, ngrid, nl, (double*)(d + o_xb) + q0 * nl, st);
                if (rc != IBS_OK) goto done;
            }
            IBS_TRY(cudaEventRecord(ev_c[c * (nsub + 1) + 1 + q], st));
            IBS_TRY(cudaStreamWaitEvent(st_d, ev_c[c * (nsub + 1) + 1 + q], 0));
            if (xbest_out) IBS_TRY(cudaMemcpyAsync(xbest_out + q0 * nl, d + o_xb + q0 * nl * 8, nq * nl * 8, cudaMemcpyDeviceToHost, st_d));
            if (xall_out) IBS_TRY(cudaMemcpyAsync(xall_out + qv0 * nl, d + o_xa + qv0 * nl * 8, nqv * nl * 8, cudaMemcpyDeviceToHost, st_d));
        }
    }
    IBS_TRY(cudaMemcpyAsync(&nbad_host, d + o_nb, 4, cudaMemcpyDeviceToHost, st_d));
    IBS_TRY(cudaEventRecord(ev_done, st_d));
    IBS_TRY(cudaStreamWaitEvent(st, ev_done, 0));          // the arena is freed (stream-ordered, on st) after the last download
    IBS_TRY(cudaStreamSynchronize(st_d));
    if (nbad_out) *nbad_out = nbad_host;
done:
#undef IBS_TRY
    if (rc != IBS_OK) { cudaStreamSynchronize(st_h); cudaStreamSynchronize(st); cudaStreamSynchronize(st_d); }
    if (d) cudaFreeAsync(d, st);
    cudaStreamSynchronize(st);
    return rc;
}

}  // extern "C"
