// Marginal stability: critical pressure-gradient factor kappa* per (field line, theta0) solve (see ibs_marginal_core.cuh).
//
//   marginal_prep_kernel   one thread per (line, point): the 48-byte record G0 G1 G2 | Cg C1 Cd of the point, h^2-scaled like the
//                          scan solver's rows, and the line's flags (bad input, c2 < 0) or-ed into one int per line
//   marginal_solve_kernel  one lane per run of CHAIN consecutive solves; every sweep streams the line's records through L1
//                          (the lanes of a line read the same addresses: broadcasts).  No shared memory and no N-dependent
//                          state, so every N the library accepts (5 .. 65 538) runs the same code.
//   marginal_tangent_kernel      one CTA per solve, after the two kernels above: d kappa* / d alpha = -x^T dK/dalpha x / qk
//                                from the records' alpha-tangent (dbase, ddPdrho of ibs_geometry_tangent_batch) at x*
//   marginal_sensitivity_kernel  one CTA per solve: qk from the caller's x*, then d kappa* / d g_j and d kappa* / d c_j per
//                                point -- what the reverse mode of K1 (ibs_geometry_adjoint_scal) consumes
// Scan-shaped batches (line = s / nth0) prepare each line once; line_of_solve batches prepare the line of every solve (the
// largest line index is on the device), with the same bits per record.
#include "ibs_common.cuh"
#include "ibs_marginal_core.cuh"

namespace ibs {

constexpr int MPREP_T = 256, MSOLVE_T = 128;

__global__ void __launch_bounds__(MPREP_T)
marginal_prep_kernel(const double* __restrict__ base, const double* __restrict__ dPdrho, const int* __restrict__ line_of_solve,
                     long long nblk, int N, double h2, double* __restrict__ rec, int* __restrict__ flags) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nblk * N) return;
    const long long blk = idx / N;
    const int j = (int)(idx - blk * N);
    const long long line = line_of_solve ? line_of_solve[blk] : blk;
    const int f = marg::prep_point(base + (size_t)line * IBS_NBASE * N, N, j, dPdrho[line], h2, rec + (size_t)idx * marg::MREC);
    if (f) atomicOr(flags + blk, f);
}

__global__ void __launch_bounds__(MSOLVE_T)
marginal_solve_kernel(const marg::MarginalArgs A, int nchain) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < nchain) marg::solve_chain(A, c);
}

int marginal_dispatch(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve, int nth0, int nsolve,
                      int N, double h, double kappa_max, double rtol, double* kappa_out, double* dlam_dkappa_out,
                      double* dkappa_dtheta0_out, double* X_out, int* info_out, cudaStream_t st) {
    const bool per_solve = line_of_solve != nullptr;
    const long long nblk = per_solve ? nsolve : ((long long)nsolve + nth0 - 1) / nth0;
    const bool want_vec = X_out || dlam_dkappa_out || dkappa_dtheta0_out;
    // one stream-ordered allocation: records | flags | X scratch (derivatives without X_out)
    const size_t rbytes = ((size_t)nblk * N * marg::MREC * sizeof(double) + 255) & ~(size_t)255;
    const size_t fbytes = ((size_t)nblk * sizeof(int) + 255) & ~(size_t)255;
    const size_t xbytes = (want_vec && !X_out) ? (size_t)nsolve * N * sizeof(double) : 0;
    char* ws = nullptr;
    IBS_CUDA_CHECK(cudaMallocAsync((void**)&ws, rbytes + fbytes + xbytes + 256, st));
    double* rec = (double*)ws;
    int* flags = (int*)(ws + rbytes);
    double* X = X_out ? X_out : (want_vec ? (double*)(ws + rbytes + fbytes) : nullptr);
    int rc = IBS_OK;
    if (cudaError_t e = cudaMemsetAsync(flags, 0, (size_t)nblk * sizeof(int), st); e != cudaSuccess) rc = cuda_fail(e, "cudaMemsetAsync");
    if (rc == IBS_OK) {
        const long long npts = nblk * N;
        marginal_prep_kernel<<<(unsigned)((npts + MPREP_T - 1) / MPREP_T), MPREP_T, 0, st>>>(base, dPdrho, line_of_solve, nblk, N, h * h, rec, flags);
        if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) rc = cuda_fail(e, "marginal_prep_kernel launch");
    }
    if (rc == IBS_OK) {
        marg::MarginalArgs A;
        A.rec = rec; A.base = base; A.dPdrho = dPdrho; A.line_flags = flags; A.theta0 = theta0; A.line_of_solve = line_of_solve;
        A.nth0 = nth0; A.nsolve = nsolve; A.N = N; A.rec_per_solve = per_solve; A.h2 = h * h; A.kmax = kappa_max; A.rtol = rtol;
        A.kappa = kappa_out; A.dlam_dkappa = dlam_dkappa_out; A.dkappa_dtheta0 = dkappa_dtheta0_out; A.X = X; A.info = info_out;
        const int nchain = (nsolve + marg::CHAIN - 1) / marg::CHAIN;
        marginal_solve_kernel<<<(unsigned)((nchain + MSOLVE_T - 1) / MSOLVE_T), MSOLVE_T, 0, st>>>(A, nchain);
        if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) rc = cuda_fail(e, "marginal_solve_kernel launch");
    }
    cudaFreeAsync(ws, st);
    return rc;
}

// ---- first-order response at kappa*: one CTA per solve, a fixed-order block sum of the per-point forms -------------------
constexpr int MRED_T = 128;

template <int K> __device__ __forceinline__ void mblock_sum(double (&v)[K]) {
    __shared__ double sm[K * (MRED_T / 32)];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = warp_sum(v[k]);
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < K; ++k) sm[warp * K + k] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double a = 0.0;
        for (int w = 0; w < MRED_T / 32; ++w) a += sm[w * K + k];
        v[k] = a;
    }
}

__device__ __forceinline__ long long line_of(const int* line_of_solve, int nth0, int s) {
    return line_of_solve ? line_of_solve[s] : s / nth0;
}
__device__ __forceinline__ bool kappa_finite(double k) { return k > 0.0 && k < INFINITY; }

// grad [s] = (d kappa* / d alpha = -qa / qk, d kappa* / d theta0 as ibs_marginal_batch gave it in dkt)
__global__ void __launch_bounds__(MRED_T)
marginal_tangent_kernel(const double* __restrict__ base, const double* __restrict__ dbase, const double* __restrict__ dPdrho,
                        const double* __restrict__ ddPdrho, const double* __restrict__ theta0, const int* __restrict__ line_of_solve,
                        int nth0, int N, double h2, const double* __restrict__ kappa, const double* __restrict__ X,
                        const double* __restrict__ dkt, double* __restrict__ grad) {
    const int s = blockIdx.x;
    const double kap = kappa[s];
    if (!kappa_finite(kap)) {                       // uniform over the CTA
        if (threadIdx.x == 0) { grad[2 * s] = NAN; grad[2 * s + 1] = dkt[s]; }
        return;
    }
    const long long line = line_of(line_of_solve, nth0, s);
    const double* b = base + (size_t)line * IBS_NBASE * N;
    const double* db = dbase + (size_t)line * IBS_NBASE * N;
    const double* x = X + (size_t)s * N;
    const double th0 = theta0[s], dP = dPdrho[line], ddP = ddPdrho[line];
    double v[2] = {0.0, 0.0};
    for (int j = threadIdx.x; j < N; j += MRED_T) {
        const marg::PointForms f = marg::point_forms(b, db, N, j, dP, ddP, h2, th0, kap, x);
        v[0] += f.qk; v[1] += f.qa;
    }
    mblock_sum<2>(v);
    if (threadIdx.x == 0) { grad[2 * s] = -v[1] / v[0]; grad[2 * s + 1] = dkt[s]; }
}

__global__ void __launch_bounds__(MRED_T)
marginal_sensitivity_kernel(const double* __restrict__ base, const double* __restrict__ dPdrho, const double* __restrict__ theta0,
                            const int* __restrict__ line_of_solve, int nth0, int N, double h2, const double* __restrict__ kappa,
                            const double* __restrict__ X, double* __restrict__ dk_dg, double* __restrict__ dk_dc) {
    const int s = blockIdx.x;
    const double kap = kappa[s];
    double* og = dk_dg + (size_t)s * N;
    double* oc = dk_dc + (size_t)s * N;
    if (!kappa_finite(kap)) {
        for (int j = threadIdx.x; j < N; j += MRED_T) { og[j] = NAN; oc[j] = NAN; }
        return;
    }
    const long long line = line_of(line_of_solve, nth0, s);
    const double* b = base + (size_t)line * IBS_NBASE * N;
    const double* x = X + (size_t)s * N;
    const double th0 = theta0[s], dP = dPdrho[line];
    double v[1] = {0.0};
    for (int j = threadIdx.x; j < N; j += MRED_T) v[0] += marg::point_forms(b, nullptr, N, j, dP, 0.0, h2, th0, kap, x).qk;
    mblock_sum<1>(v);
    const double inv = 1.0 / v[0];
    for (int j = threadIdx.x; j < N; j += MRED_T) marg::point_sensitivities(x, N, j, h2, inv, og[j], oc[j]);
}

int marginal_tangent_dispatch(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho, const double* theta0,
                              const int* line_of_solve, int nth0, int nsolve, int N, double h, double kappa_max, double rtol,
                              double* kappa_out, double* grad_out, double* X_out, int* info_out, cudaStream_t st) {
    // the solve is ibs_marginal_batch's, with d kappa* / d theta0 and X into scratch when the caller does not keep X
    const size_t tbytes = ((size_t)nsolve * sizeof(double) + 255) & ~(size_t)255;
    const size_t xbytes = X_out ? 0 : (size_t)nsolve * N * sizeof(double);
    char* ws = nullptr;
    IBS_CUDA_CHECK(cudaMallocAsync((void**)&ws, tbytes + xbytes + 256, st));
    double* dkt = (double*)ws;
    double* X = X_out ? X_out : (double*)(ws + tbytes);
    int rc = marginal_dispatch(base, dPdrho, theta0, line_of_solve, nth0, nsolve, N, h, kappa_max, rtol, kappa_out, nullptr, dkt, X,
                               info_out, st);
    if (rc == IBS_OK) {
        marginal_tangent_kernel<<<nsolve, MRED_T, 0, st>>>(base, dbase, dPdrho, ddPdrho, theta0, line_of_solve, nth0, N, h * h, kappa_out,
                                                           X, dkt, grad_out);
        if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) rc = cuda_fail(e, "marginal_tangent_kernel launch");
    }
    cudaFreeAsync(ws, st);
    return rc;
}

int marginal_sensitivity_dispatch(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve, int nth0,
                                  int nsolve, int N, double h, const double* kappa, const double* X, double* dk_dg, double* dk_dc,
                                  cudaStream_t st) {
    marginal_sensitivity_kernel<<<nsolve, MRED_T, 0, st>>>(base, dPdrho, theta0, line_of_solve, nth0, N, h * h, kappa, X, dk_dg, dk_dc);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

}  // namespace ibs
