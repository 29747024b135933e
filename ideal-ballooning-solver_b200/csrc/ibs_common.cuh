// Shared device/host helpers for the ideal-ballooning kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/ibs_b200.h"

namespace ibs {

void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);

#define IBS_CUDA_CHECK(expr)                                          \
    do {                                                              \
        cudaError_t _e = (expr);                                      \
        if (_e != cudaSuccess) return ::ibs::cuda_fail(_e, #expr);    \
    } while (0)

#define IBS_REQUIRE(cond, msg)                                        \
    do {                                                              \
        if (!(cond)) {                                                \
            ::ibs::set_error(std::string("invalid argument: ") + msg);\
            return IBS_ERR_INVALID;                                   \
        }                                                             \
    } while (0)

int num_sms();
// Index of the current device, clamped to [0, IBS_MAX_DEVICES): per-device "configured once" flags and caches are
// keyed by it (function attributes such as the dynamic shared-memory limit are per device, not per process).
constexpr int IBS_MAX_DEVICES = 64;
int current_device_slot();
// Keep stream-ordered allocations cached in the device's default memory pool between calls (by default the pool
// hands everything back to the driver at the next synchronisation, so every call would pay cudaMalloc again).
void keep_pool_cached();

// Argument block of the solver kernels (K2+K3), shared by ibs_solver.cu and ibs_api.cu.
struct SolveParams {
    // coefficient source, mode "gcf"
    const double* g; const double* c; const double* f;
    // coefficient source, mode "base"
    const double* base; const double* dPdrho; const double* theta0; const int* line_of_solve; int nth0;
    int nsolve, N; double h;
    int chain_len;      // > 1: runs of chain_len consecutive solves share a CTA and warm-start each other
    const double* lam0; const double* sigma;
    double* lam_out; double* lam_matrix_out; double* X_out; double* dX_out;
    double* g_out; double* c_out; double* f_out; int* info_out;
    // count-only mode
    const double* lam_query; int* count_out;
    // fused per-surface arg-max of a scan-shaped batch (ball_scan.py:279-295): lines_per_surface consecutive field lines form
    // a surface; best_out [nsurf][2] = (max, first flat (line-in-surface, theta0) index as a double; -1: all-zero guard,
    // -2: NaN), sigma0_out [nsurf] or null.  lines_per_surface = 0: off.
    int lines_per_surface; double* best_out; double* sigma0_out;
};

constexpr unsigned FULL = 0xffffffffu;

// ---- bit-level helpers on doubles -------------------------------------------------------------
__device__ __forceinline__ int exp_of(double v) {          // floor(log2|v|) for normal v
    return ((__double2hiint(v) >> 20) & 0x7ff) - 1023;
}
__device__ __forceinline__ double pow2i(int e) {            // 2^e, e clamped to the normal range
    e = max(-1022, min(1023, e));
    return __hiloint2double((e + 1023) << 20, 0);
}
__device__ __forceinline__ unsigned sign_word(double v) { return (unsigned)__double2hiint(v); }

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(FULL, v, src); }
// 64-bit shuffles as two explicit 32-bit shuffles (lo first): with the library overload for double ptxas allocates
// the halves in swapped order and then swaps them back with three XORs per value.
__device__ __forceinline__ double shfl_up_d(double v, int d) {
    const int lo = __shfl_up_sync(FULL, __double2loint(v), d), hi = __shfl_up_sync(FULL, __double2hiint(v), d);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_down_d(double v, int d) {
    const int lo = __shfl_down_sync(FULL, __double2loint(v), d), hi = __shfl_down_sync(FULL, __double2hiint(v), d);
    return __hiloint2double(hi, lo);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// ---- per-surface arg-max with the guards of ball_scan.py:279-295 ------------------------------------------
// (value, first flat index) maximum with the tie rule of np.where(...)[k][0] (ball_scan.py:284-285): larger value wins, equal
// values keep the smaller index; NaN is tracked separately (np.max propagates it)
__device__ __forceinline__ void best_merge(double& bv, int& bi, double ov, int oi) {
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
}
__device__ __forceinline__ void warp_best(double& bv, int& bi, int& anynan) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(FULL, bv, o);
        const int oi = __shfl_xor_sync(FULL, bi, o);
        anynan |= __shfl_xor_sync(FULL, anynan, o);
        best_merge(bv, bi, ov, oi);
    }
}
// The reduced (bv, bi, anynan) of a surface -> what the reference reports: NaN anywhere gives (NaN, -2) (np.max propagates
// it; the reference would raise), an all-zero maximum the guard's (0, -1), otherwise (max, first index); sigma0 = 0.05 for
// both guards, else 1.3 |max| + 0.05 with two roundings, like numpy (no FMA contraction).
__device__ __forceinline__ void guarded_max(double bv, int bi, int anynan, double& val, int& idx, double& sigma0) {
    if (anynan) { val = __longlong_as_double(0x7ff8000000000000LL); idx = -2; sigma0 = 0.05; }
    else if (bv == 0.0) { val = bv; idx = -1; sigma0 = 0.05; }                                      // ball_scan.py:279-282
    else { val = bv; idx = bi; sigma0 = __dadd_rn(__dmul_rn(1.3, fabs(bv)), 0.05); }                 // ball_scan.py:283-295
}

// ---- TMA bulk copy global -> shared, completion on an mbarrier -------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (unsigned)__cvta_generic_to_shared(dst)),
                 "l"(src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    const unsigned addr = (unsigned)__cvta_generic_to_shared(bar);
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    }
}

// Simpson weights of scipy.integrate.simpson with unit spacing (the reference's `simps(y)`,
// utils.py:1621).  Odd N: composite 1/3 rule.  Even N: 1/3 rule on the first N-1 points plus the
// Cartwright correction scipy >= 1.11 applies to the last interval (5/12, 2/3, -1/12).
__host__ __device__ __forceinline__ double simpson_weight(int p, int N) {
    const double third = 1.0 / 3.0;
    if (N & 1) {
        if (p == 0 || p == N - 1) return third;
        return (p & 1) ? 4.0 * third : 2.0 * third;
    }
    if (N == 2) return 0.5;
    double w = 0.0;
    const int L = N - 1;   // points covered by the basic rule
    if (p < L) w = (p == 0 || p == L - 1) ? third : ((p & 1) ? 4.0 * third : 2.0 * third);
    if (p == N - 1) w += 5.0 / 12.0;
    if (p == N - 2) w += 2.0 / 3.0;
    if (p == N - 3) w -= 1.0 / 12.0;
    return w;
}

}  // namespace ibs
