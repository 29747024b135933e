// CPU harness for the lane-per-chain code of the scan solver (csrc/ibs_scan2_core.cuh): runs solve_item2 for one solve at
// a time, the two lanes of the pair (forward chain, mirrored backward chain) one after the other, with records read
// straight from memory.  TEST INFRASTRUCTURE ONLY (tests/test_scan_core_host.py); not part of the library.
//   g++ -O2 -std=c++17 -shared -fPIC -o scan2_core_host.so tools/scan2_core_host.cpp
#include <cmath>
#include <vector>
#include <cstdio>
#include <cstdlib>
#include "scan_core_host.cpp"        // the preparation (scan_host_prep) and the two-chains-per-lane harness
#include "../ideal-ballooning-solver_b200/csrc/ibs_scan2_core.cuh"

using namespace ibs::scan2;

namespace {
struct Host2Ctx {
    const double* line_base; int N;
    const double* lvl = nullptr; int Nl = 0; int h = 0;
    long passes = 0; double cost = 0.0;
    int nev_lev[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    double* warm = nullptr;                              // warm-start records [2][nth0][WREC]: previous line | this line
    double warm_in(int token, int lev) const { return (token >= 0 && lev <= MAXLEV + 1) ? warm[token + lev] : NAN; }
    void warm_out(int token, int lev, double v) const { if (token >= 0) warm[token + lev] = v; }          // iteration passes per level (instrumentation for tools/iter_hist.py)
    void begin_pass(int lev, int Nl_, int) { lvl = line_base + (size_t)level_offset(N, lev) * REC; Nl = Nl_; }
    void wait(int) {}
    void release(int) {}
    const double* ptr(int, int q) const { return lvl + (size_t)(h ? Nl - 1 - q : q) * REC; }
    int dstep() const { return h ? -REC : REC; }
    Rec rec_k(int k) const { return load_rec(lvl + (size_t)k * REC); }
    void eval(int lev, int Nl_, int k, double th0, double lam, double& r, double& S, int& nodes) {
        const int qf = k, qb = Nl_ - 1 - k, qm = qf > qb ? qf : qb;
        h = 0; const EvalEnd f = eval_lane(*this, lev, Nl_, qf, qm, th0, lam);
        h = 1; const EvalEnd b = eval_lane(*this, lev, Nl_, qb, qm, th0, lam);
        double tk, Fk;
        row_tF(rec_k(k), th0, lam, tk, Fk);
        eval_join(f, b, tk, Fk, th0, lam, r, S, nodes);
        nev_lev[lev & 7] += 1;
        if (getenv("IBS_HOST_TRACE")) printf("  lev %d Nl %d k %d lam %.15g rho %.15g r %.3e S %.3e nodes %d\n", lev, Nl_, k, lam, lam + r / S, r, S, nodes);
        passes += 1; cost += (double)Nl_ / N;
    }
    void out1(int lev, int Nl_, int k, double th0, double lam, SolveOut& out, bool check = true) {
        const int qf = k, qb = Nl_ - 1 - k, qm = qf > qb ? qf : qb;
        Sweep f, b;
        if (check) {
            h = 0; f = out_lane<false, true>(*this, lev, Nl_, qf, qm, false, th0, lam, 0.0, 0, nullptr);
            h = 1; b = out_lane<false, true>(*this, lev, Nl_, qb, qm, true, th0, lam, 0.0, 0, nullptr);
        } else {
            h = 0; f = out_lane<false, false>(*this, lev, Nl_, qf, qm, false, th0, lam, 0.0, 0, nullptr);
            h = 1; b = out_lane<false, false>(*this, lev, Nl_, qb, qm, true, th0, lam, 0.0, 0, nullptr);
        }
        double tk, Fk;
        row_tF(rec_k(k), th0, lam, tk, Fk);
        out_join(f, b, tk, Fk, th0, lam, k, out);
        if (lev == 0) nev_lev[7] += 1;                       // first output passes on the fine level (slot 7 of the counts)
        if (getenv("IBS_HOST_TRACE")) printf("  O1 lev %d k %d lam %.15g dlt %.3e gam %.15g zmax %.3e\n", lev, k, lam, out.dlt, out.gam, out.zmax);
        passes += 1; cost += (double)Nl_ / N;
    }
    void out2(int lev, int Nl_, int k, double th0, double lam, const SolveOut& out, double* Xw) {
        const int qf = k, qb = Nl_ - 1 - k, qm = qf > qb ? qf : qb;
        const bool ok = !out.bad && out.zmax > 0.0 && out.zmax < 1e300;
        h = 0; out_lane<true, false>(*this, lev, Nl_, qf, qm, false, th0, lam, ok ? NORM_INFLATE / (out.xkf * out.zmax) : 0.0, -out.Ekf, Xw);
        h = 1; out_lane<true, false>(*this, lev, Nl_, qb, qm, true, th0, lam, ok ? NORM_INFLATE / (out.xkb * out.zmax) : 0.0, -out.Ekb, Xw);
        passes += 1; cost += (double)Nl_ / N;
    }
    bool all(bool b) const { return b; }
    bool any(bool b) const { return b; }
    int min_i(int v) const { return v; }
    int max_i(int v) const { return v; }
    int first_i(int v) const { return v; }
    void sync_mem() const {}
    double ld(const double* p) const { return *p; }
    void fixup(bool flag, double* X, double* dX, int N_, bool bad, double hh, bool want_dX) {
        if (flag) fixup_solve(*this, X, want_dX ? dX : nullptr, N_, bad, hh, 0, 1);
    }
};
std::vector<int> g_counts2;
std::vector<double> g_warm2;
}  // namespace

// iteration passes per (solve, level) of the last scan2_host_solve call: out[nsolve][8]
extern "C" long scan2_host_eval_counts(int* out) {
    for (size_t i = 0; i < g_counts2.size(); ++i) out[i] = g_counts2[i];
    return (long)g_counts2.size();
}

extern "C" int scan2_host_size_ok(int N) { return scan2_size_ok(N) ? 1 : 0; }

extern "C" long scan2_host_solve(const double* poly, const double* bounds, const double* theta0, const double* sigma, int nline,
                                 int nth0, int N, double h, double* lam_out, double* lam_matrix_out, double* X_out,
                                 double* dX_out, int* info_out) {
    const int nlev = num_levels(N), rows_total = level_offset(N, nlev + 1);
    long passes = 0; double cost = 0.0;
    g_counts2.assign((size_t)nline * nth0 * 8, 0);
    for (int line = 0; line < nline; ++line)
        for (int i = 0; i < nth0; ++i) {
            const size_t s = (size_t)line * nth0 + i;
            Host2Ctx ctx{poly + (size_t)line * rows_total * REC, N};
            // the kernel's warm start: the same theta0 of the PREVIOUS line (one sweep over the lines earlier in the kernel's
            // column order); buffer = [previous line's records | this line's records]
            const bool use_warm = !(getenv("IBS_SCAN_WARM") && atoi(getenv("IBS_SCAN_WARM")) == 0);
            const size_t half = (size_t)nth0 * WREC;
            if (line == 0 && i == 0) g_warm2.assign(2 * half, NAN);
            if (line > 0 && i == 0) { for (size_t q = 0; q < half; ++q) { g_warm2[q] = g_warm2[half + q]; g_warm2[half + q] = NAN; } }
            ctx.warm = g_warm2.data();
            const int w_in = (use_warm && line > 0) ? i * WREC : -1;
            const int w_out = use_warm ? (int)half + i * WREC : -1;
            ItemProblem P;
            P.N = N; P.nlev = nlev; P.h = h; P.U = bounds[2 * line]; P.Lb = bounds[2 * line + 1];
            P.want_X = X_out != nullptr; P.want_dX = dX_out != nullptr;
            std::vector<double> xscratch(N);
            ItemResult res;
            ColdState cold;
            solve_item2(ctx, P, theta0[s], true, sigma ? sigma[s] : 0.0, sigma != nullptr, X_out ? X_out + s * N : xscratch.data(),
                        dX_out ? dX_out + s * N : nullptr, res, cold, w_in, w_out);
            lam_out[s] = res.gam;
            if (lam_matrix_out) lam_matrix_out[s] = res.rho;
            if (info_out) info_out[s] = res.info;
            passes += ctx.passes; cost += ctx.cost;
            for (int l = 0; l < 8; ++l) g_counts2[s * 8 + l] = ctx.nev_lev[l];
        }
    g_cost = cost;
    return passes;
}
