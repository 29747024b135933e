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

// first-order response at kappa* (the per-point forms of marginal_tangent_kernel / marginal_sensitivity_kernel, summed in
// point order): grad_a [nsolve] = d kappa* / d alpha = -qa / qk; dk_dg, dk_dc [nsolve][N]
extern "C" void marginal_host_tangent(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho,
                                      const double* theta0, const int* line_of_solve, int nth0, int nsolve, int N, double h,
                                      const double* kappa, const double* X, double* grad_a) {
    for (int s = 0; s < nsolve; ++s) {
        const int line = line_of_solve ? line_of_solve[s] : s / nth0;
        const size_t o = (size_t)line * IBS_NBASE * N;
        double qk = 0.0, qa = 0.0;
        for (int j = 0; j < N; ++j) {
            const PointForms f = point_forms(base + o, dbase + o, N, j, dPdrho[line], ddPdrho[line], h * h, theta0[s], kappa[s],
                                             X + (size_t)s * N);
            qk += f.qk; qa += f.qa;
        }
        grad_a[s] = -qa / qk;
    }
}

extern "C" void marginal_host_sensitivities(const double* base, const double* dPdrho, const double* theta0, const int* line_of_solve,
                                            int nth0, int nsolve, int N, double h, const double* kappa, const double* X, double* dk_dg,
                                            double* dk_dc) {
    for (int s = 0; s < nsolve; ++s) {
        const int line = line_of_solve ? line_of_solve[s] : s / nth0;
        const double* b = base + (size_t)line * IBS_NBASE * N;
        const double* x = X + (size_t)s * N;
        double qk = 0.0;
        for (int j = 0; j < N; ++j) qk += point_forms(b, nullptr, N, j, dPdrho[line], 0.0, h * h, theta0[s], kappa[s], x).qk;
        for (int j = 0; j < N; ++j) point_sensitivities(x, N, j, h * h, 1.0 / qk, dk_dg[(size_t)s * N + j], dk_dc[(size_t)s * N + j]);
    }
}
