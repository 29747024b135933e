// Marginal stability: critical pressure-gradient factor kappa* per (field line, theta0) solve (see ibs_marginal_core.cuh).
//
//   marginal_prep_kernel   one thread per (line, point): the 48-byte record G0 G1 G2 | Cg C1 Cd of the point, h^2-scaled like the
//                          scan solver's rows, and the line's flags (bad input, c2 < 0) or-ed into one int per line
//   marginal_solve_kernel  one lane per run of CHAIN consecutive solves; every sweep streams the line's records through L1
//                          (the lanes of a line read the same addresses: broadcasts).  No shared memory and no N-dependent
//                          state, so every N the library accepts (5 .. 65 538) runs the same code.
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

}  // namespace ibs
