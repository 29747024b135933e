// K4: adjoint (Hellmann-Feynman) gradient of lambda, per-point sensitivities, and the per-surface
// arg-max of the (alpha, theta0) scan.  Replaces utils.py:1666-1680, 1707-1725 and ball_scan.py:279-295.
// These are streaming reductions (HBM-bound): one CTA per (solve[, parameter]), coalesced loads,
// warp-shuffle + shared-memory reduction.
#include "ibs_common.cuh"
#include "ibs_refine_core.cuh"

namespace ibs {

constexpr int RED_THREADS = 128;

template <int K> __device__ __forceinline__ void block_sum(double (&v)[K], double* sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = warp_sum(v[k]);
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < K; ++k) sm[warp * K + k] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double a = 0.0;
        for (int w = 0; w < nw; ++w) a += sm[w * K + k];
        v[k] = a;
    }
    __syncthreads();
}

// grad[s][q] = simps(c_p X^2)/Y1 - simps(g_p dX^2)/Y1 - lam simps(f_p X^2)/Y1   (utils.py:1676-1680)
__global__ void __launch_bounds__(RED_THREADS)
adjoint_kernel(const double* __restrict__ lam, const double* __restrict__ X, const double* __restrict__ dX,
               const double* __restrict__ f, const double* __restrict__ g_p, const double* __restrict__ c_p,
               const double* __restrict__ f_p, int nparam, int N, double* __restrict__ grad) {
    __shared__ double sm[4 * (RED_THREADS / 32)];
    const int s = blockIdx.x / nparam, q = blockIdx.x % nparam;
    const size_t row = (size_t)s * N, prow = ((size_t)s * nparam + q) * N;
    double v[4] = {0, 0, 0, 0};
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const double w = simpson_weight(j, N);
        const double x2 = __dmul_rn(X[row + j], X[row + j]), d2 = __dmul_rn(dX[row + j], dX[row + j]);
        v[0] += w * __dmul_rn(f[row + j], x2);
        v[1] += w * __dmul_rn(c_p[prow + j], x2);
        v[2] += w * __dmul_rn(g_p[prow + j], d2);
        v[3] += w * __dmul_rn(f_p[prow + j], x2);
    }
    block_sum<4>(v, sm);
    if (threadIdx.x == 0)
        grad[(size_t)s * nparam + q] = __dsub_rn(__dsub_rn(__ddiv_rn(v[1], v[0]), __ddiv_rn(v[2], v[0])),
                                                 __ddiv_rn(__dmul_rn(lam[s], v[3]), v[0]));
}

__global__ void __launch_bounds__(RED_THREADS)
sensitivity_kernel(const double* __restrict__ lam, const double* __restrict__ X, const double* __restrict__ dX,
                   const double* __restrict__ f, int N, double* __restrict__ dg, double* __restrict__ dc,
                   double* __restrict__ df) {
    __shared__ double sm[RED_THREADS / 32];
    const int s = blockIdx.x;
    const size_t row = (size_t)s * N;
    double v[1] = {0};
    for (int j = threadIdx.x; j < N; j += blockDim.x)
        v[0] += simpson_weight(j, N) * __dmul_rn(f[row + j], __dmul_rn(X[row + j], X[row + j]));
    block_sum<1>(v, sm);
    const double inv = 1.0 / v[0], l = lam[s];
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const double w = simpson_weight(j, N) * inv;
        const double x2 = X[row + j] * X[row + j], d2 = dX[row + j] * dX[row + j];
        if (dg) dg[row + j] = -w * d2;
        if (dc) dc[row + j] = w * x2;
        if (df) df[row + j] = -l * w * x2;
    }
}

// g, c, f of one field line at one point (same operation order as Coef<true> in ibs_solver.cu)
struct LineCoef {
    const double* b; int N; double dP;
    __device__ __forceinline__ void gcf(int j, double th0, double two_th0, double th0sq, double& g, double& c, double& f) const {
        const double B = b[IBS_BASE_BMAG * N + j];
        const double gp = fabs(b[IBS_BASE_GRADPAR * N + j]);
        const double cv = __dadd_rn(b[IBS_BASE_CVDRIFT * N + j], __dmul_rn(th0, b[IBS_BASE_CVDRIFT0 * N + j]));
        const double gd = __dadd_rn(__dadd_rn(b[IBS_BASE_GDS2 * N + j], __dmul_rn(two_th0, b[IBS_BASE_GDS21 * N + j])),
                                    __dmul_rn(th0sq, b[IBS_BASE_GDS22 * N + j]));
        const double gpB = __dmul_rn(gp, B);
        g = __ddiv_rn(__dmul_rn(gp, gd), B);
        c = __ddiv_rn(__dmul_rn(__dmul_rn(-1.0, dP), cv), gpB);
        f = __ddiv_rn(__ddiv_rn(gd, __dmul_rn(B, B)), gpB);
    }
};

// obj_w_grad contraction (utils.py:1666-1728) for one (alpha, theta0) point per CTA.
__global__ void __launch_bounds__(RED_THREADS)
obj_grad_kernel(const double* __restrict__ base3, const double* __restrict__ dPdrho3, const double* __restrict__ theta0,
                const double* __restrict__ lam, const double* __restrict__ X, const double* __restrict__ dX, int N,
                double del_alpha, double* __restrict__ val_out, double* __restrict__ grad_out) {
    __shared__ double sm[7 * (RED_THREADS / 32)];
    const int p = blockIdx.x;
    const size_t row = (size_t)p * N;
    LineCoef L[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        L[k].b = base3 + ((size_t)p * 3 + k) * IBS_NBASE * N;
        L[k].N = N;
        L[k].dP = dPdrho3[p * 3 + k];
    }
    const double th0 = theta0[p], two_th0 = __dmul_rn(2.0, th0), th0sq = __dmul_rn(th0, th0);
    double v[7] = {0, 0, 0, 0, 0, 0, 0};   // Y1, (c,g,f)_theta0, (c,g,f)_alpha
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const double w = simpson_weight(j, N);
        const double x2 = __dmul_rn(X[row + j], X[row + j]), d2 = __dmul_rn(dX[row + j], dX[row + j]);
        double gl, cl, fl, gc, cc, fc, gr, cr, fr;
        L[0].gcf(j, th0, two_th0, th0sq, gl, cl, fl);
        L[1].gcf(j, th0, two_th0, th0sq, gc, cc, fc);
        L[2].gcf(j, th0, two_th0, th0sq, gr, cr, fr);
        // utils.py:1669-1673
        const double* b = L[1].b;
        const double B = b[IBS_BASE_BMAG * N + j], gp = fabs(b[IBS_BASE_GRADPAR * N + j]);
        const double dgd = __dadd_rn(__dmul_rn(2.0, b[IBS_BASE_GDS21 * N + j]), __dmul_rn(two_th0, b[IBS_BASE_GDS22 * N + j]));
        const double gpB = __dmul_rn(gp, B);
        const double g_t0 = __ddiv_rn(__dmul_rn(gp, dgd), B);
        const double c_t0 = __ddiv_rn(__dmul_rn(__dmul_rn(-1.0, L[1].dP), b[IBS_BASE_CVDRIFT0 * N + j]), gpB);
        const double f_t0 = __ddiv_rn(__ddiv_rn(dgd, __dmul_rn(B, B)), gpB);
        // utils.py:1716-1718
        const double g_a = __ddiv_rn(__dsub_rn(gr, gl), del_alpha);
        const double c_a = __ddiv_rn(__dsub_rn(cr, cl), del_alpha);
        const double f_a = __ddiv_rn(__dsub_rn(fr, fl), del_alpha);
        v[0] += w * __dmul_rn(fc, x2);
        v[1] += w * __dmul_rn(c_t0, x2);
        v[2] += w * __dmul_rn(g_t0, d2);
        v[3] += w * __dmul_rn(f_t0, x2);
        v[4] += w * __dmul_rn(c_a, x2);
        v[5] += w * __dmul_rn(g_a, d2);
        v[6] += w * __dmul_rn(f_a, x2);
    }
    block_sum<7>(v, sm);
    if (threadIdx.x == 0) {
        const double l = lam[p];
        const double jt = __dsub_rn(__dsub_rn(__ddiv_rn(v[1], v[0]), __ddiv_rn(v[2], v[0])), __ddiv_rn(__dmul_rn(l, v[3]), v[0]));
        const double ja = __dsub_rn(__dsub_rn(__ddiv_rn(v[4], v[0]), __ddiv_rn(v[5], v[0])), __ddiv_rn(__dmul_rn(l, v[6]), v[0]));
        val_out[p] = -1 * l;
        grad_out[2 * p + 0] = -1 * ja;
        grad_out[2 * p + 1] = -1 * jt;
    }
}

// obj_grad_kernel with the exact alpha-derivative: one line per point and its alpha-tangent (dbase, ddPdrho from
// ibs_geometry_tangent_batch) instead of three lines.  (g, c, f)_alpha are the chain rule through LineCoef::gcf; Y1, the
// theta0 part, the thread layout and the summation order are obj_grad_kernel's, so val and grad[:, 1] are the same bits.
__global__ void __launch_bounds__(RED_THREADS)
obj_grad_tangent_kernel(const double* __restrict__ base, const double* __restrict__ dbase, const double* __restrict__ dPdrho,
                        const double* __restrict__ ddPdrho, const double* __restrict__ theta0, const double* __restrict__ lam,
                        const double* __restrict__ X, const double* __restrict__ dX, int N, double* __restrict__ val_out,
                        double* __restrict__ grad_out) {
    __shared__ double sm[7 * (RED_THREADS / 32)];
    const int p = blockIdx.x;
    const size_t row = (size_t)p * N;
    LineCoef L;
    L.b = base + (size_t)p * IBS_NBASE * N;
    L.N = N;
    L.dP = dPdrho[p];
    const double* db = dbase + (size_t)p * IBS_NBASE * N;
    const double ddP = ddPdrho[p];
    const double th0 = theta0[p], two_th0 = __dmul_rn(2.0, th0), th0sq = __dmul_rn(th0, th0);
    double v[7] = {0, 0, 0, 0, 0, 0, 0};   // Y1, (c,g,f)_theta0, (c,g,f)_alpha
    for (int j = threadIdx.x; j < N; j += blockDim.x) {
        const double w = simpson_weight(j, N);
        const double x2 = __dmul_rn(X[row + j], X[row + j]), d2 = __dmul_rn(dX[row + j], dX[row + j]);
        double gc, cc, fc;
        L.gcf(j, th0, two_th0, th0sq, gc, cc, fc);
        // utils.py:1669-1673
        const double* b = L.b;
        const double B = b[IBS_BASE_BMAG * N + j], gp = fabs(b[IBS_BASE_GRADPAR * N + j]);
        const double dgd = __dadd_rn(__dmul_rn(2.0, b[IBS_BASE_GDS21 * N + j]), __dmul_rn(two_th0, b[IBS_BASE_GDS22 * N + j]));
        const double gpB = __dmul_rn(gp, B);
        const double g_t0 = __ddiv_rn(__dmul_rn(gp, dgd), B);
        const double c_t0 = __ddiv_rn(__dmul_rn(__dmul_rn(-1.0, L.dP), b[IBS_BASE_CVDRIFT0 * N + j]), gpB);
        const double f_t0 = __ddiv_rn(__ddiv_rn(dgd, __dmul_rn(B, B)), gpB);
        // d/d alpha of g = gp gd / B, c = -dP cv / (gp B), f = gd / (B^2 gp B)
        const double cv = b[IBS_BASE_CVDRIFT * N + j] + th0 * b[IBS_BASE_CVDRIFT0 * N + j];
        const double gd = b[IBS_BASE_GDS2 * N + j] + two_th0 * b[IBS_BASE_GDS21 * N + j] + th0sq * b[IBS_BASE_GDS22 * N + j];
        const double dB = db[IBS_BASE_BMAG * N + j];
        const double dgp = (b[IBS_BASE_GRADPAR * N + j] < 0.0 ? -1.0 : 1.0) * db[IBS_BASE_GRADPAR * N + j];
        const double dcv = db[IBS_BASE_CVDRIFT * N + j] + th0 * db[IBS_BASE_CVDRIFT0 * N + j];
        const double dgdv = db[IBS_BASE_GDS2 * N + j] + two_th0 * db[IBS_BASE_GDS21 * N + j] + th0sq * db[IBS_BASE_GDS22 * N + j];
        const double rB = dB / B, rgpB = (dgp * B + gp * dB) / gpB;           // d log B, d log (gp B)
        const double g_a = (dgp * gd + gp * dgdv) / B - gc * rB;
        const double c_a = -(ddP * cv + L.dP * dcv) / gpB - cc * rgpB;
        const double f_a = dgdv / (B * B * gpB) - fc * (2.0 * rB + rgpB);
        v[0] += w * __dmul_rn(fc, x2);
        v[1] += w * __dmul_rn(c_t0, x2);
        v[2] += w * __dmul_rn(g_t0, d2);
        v[3] += w * __dmul_rn(f_t0, x2);
        v[4] += w * __dmul_rn(c_a, x2);
        v[5] += w * __dmul_rn(g_a, d2);
        v[6] += w * __dmul_rn(f_a, x2);
    }
    block_sum<7>(v, sm);
    if (threadIdx.x == 0) {
        const double l = lam[p];
        const double jt = __dsub_rn(__dsub_rn(__ddiv_rn(v[1], v[0]), __ddiv_rn(v[2], v[0])), __ddiv_rn(__dmul_rn(l, v[3]), v[0]));
        const double ja = __dsub_rn(__dsub_rn(__ddiv_rn(v[4], v[0]), __ddiv_rn(v[5], v[0])), __ddiv_rn(__dmul_rn(l, v[6]), v[0]));
        val_out[p] = -1 * l;
        grad_out[2 * p + 0] = -1 * ja;
        grad_out[2 * p + 1] = -1 * jt;
    }
}

__global__ void centre_lines_kernel(int* line, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) line[i] = 3 * i + 1;
}
__global__ void identity_lines_kernel(int* line, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) line[i] = i;
}

// Per-surface arg-max with the guards of ball_scan.py:279-295.
__global__ void __launch_bounds__(RED_THREADS)
argmax_kernel(const double* __restrict__ gamma, int ngrid, double* __restrict__ val, int* __restrict__ idx,
              double* __restrict__ sigma0, double* __restrict__ best) {
    __shared__ double sv[RED_THREADS / 32];
    __shared__ int si[RED_THREADS / 32];
    __shared__ int snan[RED_THREADS / 32];
    const int s = blockIdx.x;
    const double* gm = gamma + (size_t)s * ngrid;
    double bv = -INFINITY;
    int bi = 0x7fffffff, anynan = 0;
    for (int j = threadIdx.x; j < ngrid; j += blockDim.x) {
        const double v = gm[j];
        if (v != v) anynan = 1;
        best_merge(bv, bi, v, j);
    }
    warp_best(bv, bi, anynan);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sv[warp] = bv; si[warp] = bi; snan[warp] = anynan; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
            anynan |= snan[w];
            best_merge(bv, bi, sv[w], si[w]);
        }
        double v; int k; double sg;
        guarded_max(bv, bi, anynan, v, k, sg);
        if (val) val[s] = v;
        if (idx) idx[s] = k;
        if (sigma0) sigma0[s] = sg;
        if (best) { best[2 * s] = v; best[2 * s + 1] = (double)k; }     // packed (max, index) pair: the all-gather send slot
    }
}

// X of each surface's arg-max solve (flat index 0 when the all-zero guard fired): [ns][N]
__global__ void gather_best_kernel(const double* __restrict__ X, const int* __restrict__ idx, int ngrid, int N,
                                   double* __restrict__ out) {
    const int s = blockIdx.x;
    const int k = idx[s] < 0 ? 0 : idx[s];
    const double* src = X + ((size_t)s * ngrid + k) * N;
    for (int j = threadIdx.x; j < N; j += blockDim.x) out[(size_t)s * N + j] = src[j];
}
int launch_gather_best(const double* X, const int* idx, int ns, int ngrid, int N, double* out, cudaStream_t st) {
    if (ns == 0) return IBS_OK;
    gather_best_kernel<<<ns, 256, 0, st>>>(X, idx, ngrid, N, out);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

// Unpack the (max, index) pairs of the fused arg-max: val / idx arrays for the host, and the (line, theta0) of each
// surface's arg-max solve (flat index 0 when the all-zero guard fired) for the eigenfunction re-solve
__global__ void best_setup_kernel(const double* __restrict__ best, const double* __restrict__ theta0, int ns, int ngrid, int nth0,
                                  double* __restrict__ val_out, int* __restrict__ idx_out, int* __restrict__ line_out,
                                  double* __restrict__ th0_out) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    const int idx = (int)best[2 * s + 1];
    val_out[s] = best[2 * s];
    idx_out[s] = idx;
    const int k = idx < 0 ? 0 : idx;
    const int flat = s * ngrid + k;
    line_out[s] = flat / nth0;
    th0_out[s] = theta0[flat];
}
int launch_best_setup(const double* best, const double* theta0, int ns, int ngrid, int nth0, double* val_out, int* idx_out,
                      int* line_out, double* th0_out, cudaStream_t st) {
    if (ns == 0) return IBS_OK;
    best_setup_kernel<<<(ns + 127) / 128, 128, 0, st>>>(best, theta0, ns, ngrid, nth0, val_out, idx_out, line_out, th0_out);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

// ---- batched refinement of the coarse maxima (ball_scan.py:305-314): one thread per surface -----------------------------
// Consumes the batched obj_w_grad evaluation of every problem's trial point, advances the problems (see ibs_refine_core.cuh)
// and writes the next trial points in the layout the evaluation takes: alphas3 [n][3] = (a - del/2, a, a + del/2)
// (utils.py:1641-1646) and theta0 [n].
__global__ void refine_init_kernel(double* __restrict__ state, int n, const double* __restrict__ a0, const double* __restrict__ t0,
                                   double alo, double ahi, double tlo, double thi, double del_alpha, double* __restrict__ alphas3,
                                   double* __restrict__ theta0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    refine::State s;
    refine::init(s, a0[i], t0[i], alo, ahi, tlo, thi);
    double* o = state + (size_t)i * refine::NSTATE;
    const double* src = reinterpret_cast<const double*>(&s);
    for (int k = 0; k < refine::NSTATE; ++k) o[k] = src[k];
    alphas3[3 * i] = s.xt[0] - 0.5 * del_alpha; alphas3[3 * i + 1] = s.xt[0]; alphas3[3 * i + 2] = s.xt[0] + 0.5 * del_alpha;
    theta0[i] = s.xt[1];
}
__global__ void refine_step_kernel(double* __restrict__ state, int n, const double* __restrict__ val, const double* __restrict__ grad,
                                   const int* __restrict__ info, refine::Options opt, double del_alpha, double* __restrict__ alphas3,
                                   double* __restrict__ theta0, int* __restrict__ nactive) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool active = false;
    if (i < n) {
        refine::State s;
        double* o = state + (size_t)i * refine::NSTATE;
        double* dst = reinterpret_cast<double*>(&s);
        for (int k = 0; k < refine::NSTATE; ++k) dst[k] = o[k];
        const bool failed = info && ((info[i] >> 16) & (IBS_FLAG_NOT_CONVERGED | IBS_FLAG_BAD_INPUT));
        refine::consume(s, val[i], grad[2 * i], grad[2 * i + 1], failed, opt);
        for (int k = 0; k < refine::NSTATE; ++k) o[k] = dst[k];
        alphas3[3 * i] = s.xt[0] - 0.5 * del_alpha; alphas3[3 * i + 1] = s.xt[0]; alphas3[3 * i + 2] = s.xt[0] + 0.5 * del_alpha;
        theta0[i] = s.xt[1];
        active = (int)s.status != refine::ST_DONE;
    }
    const unsigned m = __ballot_sync(FULL, active);
    if (nactive && (threadIdx.x & 31) == 0 && m) atomicAdd(nactive, __popc(m));
}
int launch_refine_init(double* state, int n, const double* a0, const double* t0, double alo, double ahi, double tlo, double thi,
                       double del_alpha, double* alphas3, double* theta0, cudaStream_t st) {
    if (n == 0) return IBS_OK;
    refine_init_kernel<<<(n + 127) / 128, 128, 0, st>>>(state, n, a0, t0, alo, ahi, tlo, thi, del_alpha, alphas3, theta0);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_refine_step(double* state, int n, const double* val, const double* grad, const int* info, double ftol, double gtol,
                       int maxiter, double del_alpha, double* alphas3, double* theta0, int* nactive, cudaStream_t st) {
    if (n == 0) return IBS_OK;
    if (nactive) IBS_CUDA_CHECK(cudaMemsetAsync(nactive, 0, sizeof(int), st));
    refine::Options o; o.ftol = ftol; o.gtol = gtol; o.maxiter = maxiter;
    refine_step_kernel<<<(n + 127) / 128, 128, 0, st>>>(state, n, val, grad, info, o, del_alpha, alphas3, theta0, nactive);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

int launch_adjoint(const double* lam, const double* X, const double* dX, const double* f, const double* g_p,
                   const double* c_p, const double* f_p, int nsolve, int nparam, int N, double* grad,
                   cudaStream_t st) {
    if (nsolve * nparam == 0) return IBS_OK;
    adjoint_kernel<<<nsolve * nparam, RED_THREADS, 0, st>>>(lam, X, dX, f, g_p, c_p, f_p, nparam, N, grad);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_sensitivity(const double* lam, const double* X, const double* dX, const double* f, int nsolve, int N,
                       double* dg, double* dc, double* df, cudaStream_t st) {
    if (nsolve == 0) return IBS_OK;
    sensitivity_kernel<<<nsolve, RED_THREADS, 0, st>>>(lam, X, dX, f, N, dg, dc, df);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_obj_grad(const double* base3, const double* dPdrho3, const double* theta0, const double* lam,
                    const double* X, const double* dX, int npoint, int N, double del_alpha, double* val,
                    double* grad, cudaStream_t st) {
    if (npoint == 0) return IBS_OK;
    obj_grad_kernel<<<npoint, RED_THREADS, 0, st>>>(base3, dPdrho3, theta0, lam, X, dX, N, del_alpha, val, grad);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_obj_grad_tangent(const double* base, const double* dbase, const double* dPdrho, const double* ddPdrho, const double* theta0,
                            const double* lam, const double* X, const double* dX, int npoint, int N, double* val, double* grad,
                            cudaStream_t st) {
    if (npoint == 0) return IBS_OK;
    obj_grad_tangent_kernel<<<npoint, RED_THREADS, 0, st>>>(base, dbase, dPdrho, ddPdrho, theta0, lam, X, dX, N, val, grad);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_centre_lines(int* line, int n, cudaStream_t st) {
    if (n == 0) return IBS_OK;
    centre_lines_kernel<<<(n + 255) / 256, 256, 0, st>>>(line, n);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_identity_lines(int* line, int n, cudaStream_t st) {
    if (n == 0) return IBS_OK;
    identity_lines_kernel<<<(n + 255) / 256, 256, 0, st>>>(line, n);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_argmax(const double* gamma, int ns, int ngrid, double* val, int* idx, double* sigma0, cudaStream_t st) {
    if (ns == 0) return IBS_OK;
    argmax_kernel<<<ns, RED_THREADS, 0, st>>>(gamma, ngrid, val, idx, sigma0, nullptr);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
int launch_argmax_packed(const double* gamma, int ns, int ngrid, double* best, double* sigma0, cudaStream_t st) {
    if (ns == 0) return IBS_OK;
    argmax_kernel<<<ns, RED_THREADS, 0, st>>>(gamma, ngrid, nullptr, nullptr, sigma0, best);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}

}  // namespace ibs
