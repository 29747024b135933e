// CPU harness for the lane code of the scan solver (csrc/ibs_scan_core.cuh): runs solve_item for one lane at a
// time with records read straight from memory.  TEST INFRASTRUCTURE ONLY (tests/test_scan_core_host.py): it checks
// the per-lane arithmetic, indices and iteration logic without a GPU; it is not part of the library and nothing in
// the product path calls it.
//   g++ -O2 -std=c++17 -shared -fPIC -o scan_core_host.so tools/scan_core_host.cpp
#include <algorithm>
#include <cmath>
#include <vector>

#include "../ideal-ballooning-solver_b200/csrc/ibs_scan_core.cuh"

using namespace ibs::scan;
static double g_cost = 0.0;

namespace {
struct HostCtx {
    const double* line_base; int N;
    const double* lvl = nullptr; int Nl = 0, cur = 0;
    long evals = 0; double cost = 0.0;
    void begin_pass(int lev, int Nl_, int, int) { lvl = line_base + (size_t)level_offset(N, lev) * REC; Nl = Nl_; cur = 0; evals += 1; cost += (double)Nl_ / N; }
    void wait(int s) { cur = s; }
    const double* frec(int i) const { return lvl + (size_t)(TR * cur + i) * REC; }
    const double* brec(int i) const { return lvl + (size_t)(Nl - 1 - (TR * cur + i)) * REC; }
    void release(int) {}
    bool all(bool b) const { return b; }
    bool any(bool b) const { return b; }
    int min_i(int v) const { return v; }
    int max_i(int v) const { return v; }
    int first_i(int v) const { return v; }
    void sync_mem() const {}
    std::vector<double> scr = std::vector<double>(4096);
    double* scratch() { return scr.data(); }
    double ld(const double* p) const { return *p; }
    int ldi(const int* p) const { return *p; }
    void fixup(bool flag, double* X, double* dX, int N_, bool bad, double h, bool want_dX) {
        if (flag) fixup_solve(*this, X, want_dX ? dX : nullptr, N_, bad, h, 0, 1);
    }
};
}  // namespace

// Host version of the preparation: records of all levels of every line + per-line bounds (U, Lb).
// base: [nline][8][N] (IBS_BASE_* order), theta0: [nline * nth0].  poly: [nline][rows_total][6], bounds: [nline][2].
extern "C" int scan_host_rows_total(int N) { return level_offset(N, num_levels(N) + 1); }
extern "C" int scan_host_num_levels(int N) { return num_levels(N); }

extern "C" void scan_host_prep(const double* base, const double* dPdrho, const double* theta0, int nline, int nth0, int N,
                               double h, double* poly, double* bounds) {
    const int nlev = num_levels(N), rows_total = level_offset(N, nlev + 1);
    const double h2 = h * h;
    for (int line = 0; line < nline; ++line) {
        const double* b = base + (size_t)line * 8 * N;
        double t0 = 1e300, t1 = -1e300;
        for (int i = 0; i < nth0; ++i) { t0 = std::min(t0, theta0[(size_t)line * nth0 + i]); t1 = std::max(t1, theta0[(size_t)line * nth0 + i]); }
        std::vector<Rec> recs(N);
        double gmax = 0.0;
        for (int j = 0; j < N; ++j) {
            recs[j] = raw_record(b[0 * N + j], b[1 * N + j], b[2 * N + j], b[3 * N + j], b[4 * N + j], b[5 * N + j], b[6 * N + j], dPdrho[line], h2);
            double gmn, gmx, cmn, cmx;
            record_ranges(recs[j], t0, t1, gmn, gmx, cmn, cmx);
            if (gmx > gmax) gmax = gmx;
        }
        const double sg = (gmax > 0.0 && gmax < 1e300) ? pow2(-exp_max2(gmax, 0.0)) : 1.0;
        double U = -1e300, minC = 1e300, maxg = 0.0, minF = 1e300, maxF = 0.0;
        double* out = poly + (size_t)line * rows_total * REC;
        for (int j = 0; j < N; ++j) {
            Rec r = recs[j];
            r.G0 *= sg; r.G1 *= sg; r.G2 *= sg; r.C0 *= sg; r.C1 *= sg;
            double gmn, gmx, cmn, cmx;
            record_ranges(r, t0, t1, gmn, gmx, cmn, cmx);
            maxg = std::max(maxg, gmx);
            if (j >= 1 && j <= N - 2) {
                const double Fmin = gmn * r.R, Fmax = gmx * r.R;
                U = std::max(U, cmx >= 0.0 ? cmx / Fmin : cmx / Fmax);
                minC = std::min(minC, cmn); minF = std::min(minF, Fmin); maxF = std::max(maxF, Fmax);
            }
            for (int lev = 0; lev <= nlev; ++lev) {
                if (j % (1 << lev)) break;
                const double f4 = (double)(1 << (2 * lev));
                double* o = out + ((size_t)level_offset(N, lev) + (j >> lev)) * REC;
                o[0] = r.G0; o[1] = r.G1; o[2] = r.G2; o[3] = r.C0 * f4; o[4] = r.C1 * f4; o[5] = r.R * f4;
            }
        }
        U = U + 1e-12 * std::fabs(U) + 1e-300;
        const double numer = minC - 8.0 * maxg;
        bounds[2 * line + 0] = U;
        bounds[2 * line + 1] = 1.000001 * ((numer < 0.0) ? numer / minF : numer / maxF) - 1e-300;
    }
}

extern "C" long scan_host_solve(const double* poly, const double* bounds, const double* theta0, const double* sigma, int nline,
                                int nth0, int N, double h, double* lam_out, double* lam_matrix_out, double* X_out,
                                double* dX_out, int* info_out) {
    const int nlev = num_levels(N), rows_total = level_offset(N, nlev + 1);
    long passes = 0; double cost = 0.0;
    for (int line = 0; line < nline; ++line)
        for (int i = 0; i < nth0; ++i) {
            const size_t s = (size_t)line * nth0 + i;
            HostCtx ctx{poly + (size_t)line * rows_total * REC, N};
            ItemProblem P;
            P.N = N; P.nlev = nlev; P.h = h; P.U = bounds[2 * line]; P.Lb = bounds[2 * line + 1];
            P.want_X = X_out != nullptr; P.want_dX = dX_out != nullptr;
            std::vector<double> xscratch(N);
            ItemResult res;
            ColdState cold;
            solve_item(ctx, P, theta0[s], true, sigma ? sigma[s] : 0.0, sigma != nullptr, X_out ? X_out + s * N : xscratch.data(),
                       dX_out ? dX_out + s * N : nullptr, res, cold);
            lam_out[s] = res.gam;
            if (lam_matrix_out) lam_matrix_out[s] = res.rho;
            if (info_out) info_out[s] = res.info;
            passes += ctx.evals; cost += ctx.cost;
        }
    g_cost = cost;
    return passes;
}
extern "C" double scan_host_last_cost() { return g_cost; }
