// CPU harness for the lane code of the marginal-stability kernel (csrc/ibs_marginal_core.cuh): the same record preparation,
// sweeps, root finder and null-vector outputs, one lane after the other.  TEST INFRASTRUCTURE ONLY
// (tests/test_marginal_core_host.py); not part of the library.
//   g++ -O2 -std=c++17 -shared -fPIC -o marginal_core_host.so tools/marginal_core_host.cpp
#include <cmath>
#include <vector>
#include "../ideal-ballooning-solver_b200/csrc/ibs_marginal_core.cuh"

using namespace ibs::marg;

// records [nline][N][MREC] and per-line flags of base [nline][8][N]
extern "C" void marginal_host_prep(const double* base, const double* dPdrho, int nline, int N, double h, double* rec, int* line_flags) {
    for (int l = 0; l < nline; ++l) {
        int f = 0;
        for (int j = 0; j < N; ++j)
            f |= prep_point(base + (size_t)l * IBS_NBASE * N, N, j, dPdrho[l], h * h, rec + ((size_t)l * N + j) * MREC);
        line_flags[l] = f;
    }
}

extern "C" void marginal_host_solve(const double* rec, const double* base, const double* dPdrho, const int* line_flags,
                                    const double* theta0, const int* line_of_solve, int nth0, int nsolve, int N, double h,
                                    double kappa_max, double rtol, double* kappa, double* dlam, double* dkt, double* X, int* info) {
    MarginalArgs A{rec, base, dPdrho, line_flags, theta0, line_of_solve, nth0, nsolve, N, false, h * h, kappa_max, rtol, kappa, dlam, dkt, X, info};
    for (int c = 0; c * CHAIN < nsolve; ++c) solve_chain(A, c);
}

// one sweep at (kappa, lam = 0) of one line's records: count, d log|det K| / d kappa
extern "C" int marginal_host_sweep(const double* rec, int N, double th0, double kappa, double* phi) {
    const SweepOut s = sweep<true>(rec, N, th0, kappa);
    *phi = s.phi;
    return s.bad ? -1 : s.count;
}
