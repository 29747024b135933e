// K2+K3 for scan-shaped batches: lane-per-solve kernel (see ibs_scan_core.cuh for the algorithm).
//
// Replaces the theta0 loop around gamma_ball_full (/root/reference/ball_scan.py:262-274, utils.py:1550-1624) for
// batches in which every field line is solved for a row of theta0 values.
//   scan_prep_kernel   one CTA per field line: the six theta0-independent coefficient rows of the line as 48-byte
//                      records, for the fine grid and up to four coarser ones (every 2nd/4th/8th/16th point), scaled by
//                      a power of two so that max g ~ 1; bounds of the spectrum valid for the line's whole theta0 range
//   scan_solve_kernel  persistent warps; a warp takes (line, group of 32 theta0) items from a global counter.
//                      The records are streamed through a per-warp ring of shared-memory tiles with TMA bulk copies
//                      (cp.async.bulk + mbarrier, a ring of 3 stages: two ahead); every lane reads the SAME record
//                      (broadcast LDS.128) and advances its own solve.  No shuffles in the passes, no block barriers, no
//                      per-solve set-up; the state no loop touches lives in shared memory (one block per thread); HBM
//                      traffic is the records once (they stay in L2 for the ~23 passes of an item) plus the outputs.
#include <cmath>
#include <cstdlib>

#include "ibs_common.cuh"
#include "ibs_scan_core.cuh"
#include "ibs_scan2_core.cuh"

namespace ibs {
using namespace scan;

#ifndef IBS_SCAN_NSTAGE
#define IBS_SCAN_NSTAGE 3
#endif
constexpr int SC_NSTAGE = IBS_SCAN_NSTAGE;         // pipeline stages per warp
constexpr int SC_TILE = TR * REC;                  // doubles per tile (1536 B)
constexpr int SC_STAGE = 2 * SC_TILE;              // forward + backward tile
constexpr int SC_RING = SC_NSTAGE * SC_STAGE;      // doubles per warp (9 KB with 3 stages)
#ifndef IBS_SCAN_WARPS
#define IBS_SCAN_WARPS 4
#endif
constexpr int SC_WARPS = IBS_SCAN_WARPS;           // warps per CTA (they never synchronise with each other)
#ifndef IBS_SCAN_CTAS1
#define IBS_SCAN_CTAS1 2      // CTAs per SM scan_solve_kernel is compiled for (register cap 65536 / (128 * CTAS))
#endif

struct ScanParams {
    const double* poly;       // [nline][rows_total][REC]
    const double* bounds;     // [nline][2]: U, Lb
    const int* line_safe;     // [nline]: 1 = every row of the line has valid coefficients on the whole theta0 range (scan_prep_kernel)
    const double* theta0;     // [nline * nth0]
    const double* sigma;      // nullable
    int nline, nth0, N, nlev, rows_total, groups, nitems;
    int lc, rounds;           // lane-per-chain kernel: lines per round and rounds of the column order (nitems = rounds * lc * groups, padded)
    double h;
    double* lam_out; double* lam_matrix_out; double* X_out; double* dX_out; int* info_out;
    double* warm; unsigned* warm_flag;     // lane-per-chain kernel: [nline * groups][16][WREC] warm-start records handed to the next line, [nline * groups] ready flags (zeroed); null: off
    double* X_rows;           // where the eigenfunctions go: X_out, or scratch when only dX is wanted (null: no eigenfunction output)
    unsigned* counter;
    // fused per-surface arg-max (ball_scan.py:279-295); items_per_surface = 0: off
    int items_per_surface, lines_per_surface;
    double* item_val; int* item_idx;       // [nitems]: best of each (line, theta0-group) item; idx = -2: the item holds a NaN
    unsigned* surf_count;                  // [nsurf], zeroed: items of the surface that have finished
    double* best_out; double* sigma0_out;  // [nsurf][2] packed (max, flat index as a double), [nsurf] (nullable)
};

// ---- fused arg-max: each item's best (value, index) goes to its slot; the LAST item of a surface to finish (prev = the
// surface's count of finished items before this one, from lane 0) reduces the slots and writes the guarded result
__device__ __forceinline__ void surface_argmax_last(const ScanParams& p, int surf, unsigned prev, int lane) {
    prev = __shfl_sync(FULL, prev, 0);
    if (prev != (unsigned)p.items_per_surface - 1u) return;
    __threadfence();
    double bv = -INFINITY; int bi = 0x7fffffff, anynan = 0;
    const int i0 = surf * p.items_per_surface;
    for (int i = lane; i < p.items_per_surface; i += 32) {
        const double v = __ldcg(p.item_val + i0 + i);
        const int k = __ldcg(p.item_idx + i0 + i);
        if (k == -2) anynan = 1; else best_merge(bv, bi, v, k);
    }
    warp_best(bv, bi, anynan);
    if (lane == 0) {
        double val, sg; int idx;
        guarded_max(bv, bi, anynan, val, idx, sg);
        p.best_out[2 * surf] = val; p.best_out[2 * surf + 1] = (double)idx;
        if (p.sigma0_out) p.sigma0_out[surf] = sg;
    }
}

// ---- device context: record streaming + warp votes --------------------------------------------------
struct DevCtx {
    double* ring; uint64_t* bars; unsigned parity; int lane;
    const double* line_base; int N;
    const double* lvl; int Nl, nst, qf_end, qb_end;
    const double* tf; const double* tb;

    __device__ __forceinline__ void issue(int s) {          // lane 0
        const int slot = s % SC_NSTAGE;
        double* dstf = ring + slot * SC_STAGE;
        double* dstb = dstf + SC_TILE;
        const int f0 = TR * s;
        const int fn = (f0 <= qf_end) ? min(TR, Nl - f0) : 0;
        const int b1 = Nl - TR * s;
        const int b0 = max(0, b1 - TR);
        const int bn = (TR * s <= qb_end) ? (b1 - b0) : 0;
        mbar_expect_tx(&bars[slot], (unsigned)((fn + bn) * REC * sizeof(double)));
        if (fn) tma_bulk_g2s(dstf, lvl + (size_t)f0 * REC, (unsigned)(fn * REC * sizeof(double)), &bars[slot]);
        if (bn) tma_bulk_g2s(dstb + (TR - bn) * REC, lvl + (size_t)b0 * REC, (unsigned)(bn * REC * sizeof(double)), &bars[slot]);
    }
    __device__ __forceinline__ void begin_pass(int lev, int Nl_, int k, int nst_) {
        lvl = line_base + (size_t)level_offset(N, lev) * REC;
        Nl = Nl_; nst = nst_; qf_end = k; qb_end = Nl_ - 1 - k;
        __syncwarp();
        if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            const int n0 = nst < SC_NSTAGE ? nst : SC_NSTAGE;
            for (int s = 0; s < n0; ++s) issue(s);
        }
    }
    __device__ __forceinline__ void wait(int s) {
        const int slot = s % SC_NSTAGE;
        // bounded spin: a pipeline bug must trap, not hang the device
        const unsigned addr = (unsigned)__cvta_generic_to_shared(&bars[slot]), par = (parity >> slot) & 1u;
        unsigned done = 0, spins = 0;
        while (!done) {
            asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                         : "=r"(done) : "r"(addr), "r"(par) : "memory");
            if (!done && ++spins > (1u << 24)) __trap();
        }
        parity ^= 1u << slot;
        tf = ring + slot * SC_STAGE;
        tb = tf + SC_TILE;
    }
    __device__ __forceinline__ const double* frec(int i) const { return tf + i * REC; }
    __device__ __forceinline__ const double* brec(int i) const { return tb + (TR - 1 - i) * REC; }
    __device__ __forceinline__ void release(int s) {
        __syncwarp();                                        // every lane has consumed the stage
        if (lane == 0 && s + SC_NSTAGE < nst) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(s + SC_NSTAGE);
        }
    }
    __device__ __forceinline__ bool all(bool b) const { return __all_sync(FULL, b); }
    __device__ __forceinline__ bool any(bool b) const { return __any_sync(FULL, b); }
    __device__ __forceinline__ int min_i(int v) const { return __reduce_min_sync(FULL, v); }
    __device__ __forceinline__ int max_i(int v) const { return __reduce_max_sync(FULL, v); }
    __device__ __forceinline__ int first_i(int v) const {   // v of the first lane with v >= 0 (at least one exists)
        const unsigned m = __ballot_sync(FULL, v >= 0);
        return __shfl_sync(FULL, v, m ? (__ffs(m) - 1) : 0);
    }
    // the fix-up reads rows that OTHER lanes of the warp have written: L2 loads after a warp-level fence
    __device__ __forceinline__ void sync_mem() const { __syncwarp(); }
    __device__ __forceinline__ double ld(const double* p) const { return __ldcg(p); }
    // zero-fill invalid solves / form dX of the flagged solves: one solve at a time, its rows dealt out over the 32 lanes
    __device__ __forceinline__ void fixup(bool flag, double* Xrow, double* dXrow, int N_, bool bad, double h, bool want_dX) {
        __syncwarp();
        unsigned m = __ballot_sync(FULL, flag);
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const bool bd = __shfl_sync(FULL, (int)bad, l) != 0;
            double* X = reinterpret_cast<double*>(__shfl_sync(FULL, reinterpret_cast<unsigned long long>(Xrow), l));
            double* dX = reinterpret_cast<double*>(__shfl_sync(FULL, reinterpret_cast<unsigned long long>(dXrow), l));
            fixup_solve(*this, X, want_dX ? dX : nullptr, N_, bd, h, lane, 32);
        }
        __syncwarp();
    }
};

__global__ void __launch_bounds__(SC_WARPS * 32, IBS_SCAN_CTAS1)
scan_solve_kernel(const ScanParams p) {
    extern __shared__ __align__(128) double sc_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    DevCtx ctx;
    ctx.ring = sc_smem + warp * SC_RING;
    ctx.bars = reinterpret_cast<uint64_t*>(sc_smem + SC_WARPS * SC_RING) + warp * SC_NSTAGE;
    // the thread's block of cold state (odd stride in doubles: conflict-free across the lanes of a warp)
    ColdState& cold = *reinterpret_cast<ColdState*>(sc_smem + SC_WARPS * SC_RING + SC_WARPS * SC_NSTAGE + (size_t)threadIdx.x * COLD_STRIDE);
    ctx.parity = 0; ctx.lane = lane; ctx.N = p.N;
    if (lane == 0) {
        for (int s = 0; s < SC_NSTAGE; ++s) mbar_init(&ctx.bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const int N = p.N;
    for (;;) {
        int item = 0;
        if (lane == 0) item = (int)atomicAdd(p.counter, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= p.nitems) break;
        const int line = item / p.groups, grp = item - line * p.groups;
        const int idx = grp * 32 + lane;
        const bool act = idx < p.nth0;
        const size_t sidx = (size_t)line * p.nth0 + (act ? idx : p.nth0 - 1);
        const double th0 = p.theta0[sidx];
        const double sg = p.sigma ? p.sigma[sidx] : 0.0;
        double* Xrow = (act && p.X_rows) ? p.X_rows + sidx * N : nullptr;
        double* dXrow = (act && p.dX_out) ? p.dX_out + sidx * N : nullptr;
        ItemProblem P;
        P.N = N; P.nlev = p.nlev; P.h = p.h; P.U = p.bounds[2 * line]; P.Lb = p.bounds[2 * line + 1];
        P.want_X = p.X_rows != nullptr; P.want_dX = p.dX_out != nullptr;
        ctx.line_base = p.poly + (size_t)line * p.rows_total * REC;
        ItemResult res;
        solve_item(ctx, P, th0, act, sg, p.sigma != nullptr, Xrow, dXrow, res, cold);
        if (act) {
            p.lam_out[sidx] = res.gam;
            if (p.lam_matrix_out) p.lam_matrix_out[sidx] = res.rho;
            if (p.info_out) p.info_out[sidx] = res.info;
        }
        if (p.items_per_surface > 0) {
            const int surf = line / p.lines_per_surface;
            double bv = -INFINITY; int bi = 0x7fffffff, anynan = 0;
            if (act) {
                const double v = res.gam;
                if (v != v) anynan = 1;
                best_merge(bv, bi, v, (line - surf * p.lines_per_surface) * p.nth0 + idx);
            }
            warp_best(bv, bi, anynan);
            unsigned prev = 0;
            if (lane == 0) {
                p.item_val[item] = bv;
                p.item_idx[item] = anynan ? -2 : bi;
                __threadfence();
                prev = atomicAdd(&p.surf_count[surf], 1u);
            }
            surface_argmax_last(p, surf, prev, lane);
        }
    }
}

// ---- lane-per-chain kernel (ibs_scan2_core.cuh): 16 solves per warp, lane = 16 h + i runs chain h of solve i ---------------
#ifndef IBS_SCAN2_CTAS
#define IBS_SCAN2_CTAS 4          // CTAs of 4 warps per SM the kernel is compiled for (register cap 65536 / (128 * CTAS))
#endif
constexpr int S2_TILE = scan2::T0 * REC;           // doubles per tile (35 records)
constexpr int S2_STAGE = 2 * S2_TILE;              // ascending tile (forward lanes) + descending tile (backward lanes)
constexpr int S2_RING = SC_NSTAGE * S2_STAGE;      // doubles per warp (10 KB with 3 stages)

struct Dev2Ctx {
    double* ring; uint64_t* bars; unsigned parity; int lane, h;
    const double* line_base; int N;
    const double* lvl; int Nl, nst;
    double* warm;                                            // warm-start records (global memory); tokens are element offsets

    __device__ __forceinline__ double warm_in(int token, int lev) const {
        return (token >= 0 && lev <= MAXLEV + 1) ? __ldcg(warm + token + lev) : __longlong_as_double(0x7ff8000000000000LL);
    }
    __device__ __forceinline__ void warm_out(int token, int lev, double v) const {
        if (token >= 0 && h == 0) __stcg(warm + token + lev, v);
    }
    __device__ __forceinline__ void issue(int s) {          // lane 0: both tiles of stage s
        const int slot = s % SC_NSTAGE;
        double* dstA = ring + slot * S2_STAGE;
        double* dstD = dstA + S2_TILE;
        const int f0 = scan2::stage_first(s), len = scan2::stage_len(s, Nl);
        mbar_expect_tx(&bars[slot], (unsigned)(2 * len * REC * sizeof(double)));
        tma_bulk_g2s(dstA, lvl + (size_t)f0 * REC, (unsigned)(len * REC * sizeof(double)), &bars[slot]);
        tma_bulk_g2s(dstD, lvl + (size_t)(Nl - f0 - len) * REC, (unsigned)(len * REC * sizeof(double)), &bars[slot]);
    }
    __device__ __forceinline__ void begin_pass(int lev, int Nl_, int q_max) {
        lvl = line_base + (size_t)level_offset(N, lev) * REC;
        Nl = Nl_; nst = scan2::stage_of(q_max + 2) + 1;
        __syncwarp();
        if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            const int n0 = nst < SC_NSTAGE ? nst : SC_NSTAGE;
            for (int s = 0; s < n0; ++s) issue(s);
        }
    }
    __device__ __forceinline__ void wait(int s) {
        const int slot = s % SC_NSTAGE;
        const unsigned addr = (unsigned)__cvta_generic_to_shared(&bars[slot]), par = (parity >> slot) & 1u;
        unsigned done = 0, spins = 0;
        while (!done) {
            asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                         : "=r"(done) : "r"(addr), "r"(par) : "memory");
            if (!done && ++spins > (1u << 24)) __trap();        // a pipeline bug must trap, not hang the device
        }
        parity ^= 1u << slot;
    }
    // my record of step q inside stage s: ascending tile for the forward chain, descending tile read backwards for the mirrored one
    __device__ __forceinline__ const double* ptr(int s, int q) const {
        const double* t = ring + (s % SC_NSTAGE) * S2_STAGE;
        const int i = q - scan2::stage_first(s);
        return h ? t + S2_TILE + (scan2::stage_len(s, Nl) - 1 - i) * REC : t + i * REC;
    }
    __device__ __forceinline__ int dstep() const { return h ? -REC : REC; }
    __device__ __forceinline__ void release(int s) {
        __syncwarp();
        if (lane == 0 && s + SC_NSTAGE < nst) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(s + SC_NSTAGE);
        }
    }
    __device__ __forceinline__ double xd(double v) const { return __shfl_xor_sync(FULL, v, 16); }
    __device__ __forceinline__ int xi(int v) const { return __shfl_xor_sync(FULL, v, 16); }
    __device__ __forceinline__ Rec rec_k(int k) const {        // record of the matching row for the join of a pass (global memory; L2)
        const double2* q = reinterpret_cast<const double2*>(lvl + (size_t)k * REC);
        const double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
        Rec r; r.G0 = a.x; r.G1 = a.y; r.G2 = b.x; r.C0 = b.y; r.C1 = c.x; r.R = c.y;
        return r;
    }
    // ---- the passes of solve_item2: my chain, the partner's end state by shuffle, the join
    __device__ __forceinline__ void eval(int lev, int Nl_, int k, double th0, double lam, double& r, double& S, int& nodes) {
        const int qf = k, qb = Nl_ - 1 - k;
        const scan2::EvalEnd me = scan2::eval_lane(*this, lev, Nl_, h ? qb : qf, qf > qb ? qf : qb, th0, lam);
        scan2::EvalEnd ot;
        ot.X = xd(me.X); ot.W = xd(me.W); ot.S = xd(me.S); ot.nodes = xi(me.nodes);
        double tk, Fk;
        scan2::row_tF(rec_k(k), th0, lam, tk, Fk);
        scan2::eval_join(h ? ot : me, h ? me : ot, tk, Fk, th0, lam, r, S, nodes);
    }
    __device__ __forceinline__ void out1(int lev, int Nl_, int k, double th0, double lam, SolveOut& out, bool check) {
        const int qf = k, qb = Nl_ - 1 - k;
        // (check is warp-uniform: a property of the line)
        const Sweep me = check ? scan2::out_lane<false, true>(*this, lev, Nl_, h ? qb : qf, qf > qb ? qf : qb, h != 0, th0, lam, 0.0, 0, nullptr)
                               : scan2::out_lane<false, false>(*this, lev, Nl_, h ? qb : qf, qf > qb ? qf : qb, h != 0, th0, lam, 0.0, 0, nullptr);
        Sweep ot;
        ot.x = xd(me.x); ot.w = xd(me.w); ot.E = xi(me.E); ot.W2 = xd(me.W2); ot.W3 = xd(me.W3); ot.W4 = xd(me.W4); ot.gp = xd(me.gp); ot.gpp = xd(me.gpp);
        ot.a0e = xd(me.a0e); ot.a0o = xd(me.a0o); ot.a1e = xd(me.a1e); ot.a1o = xd(me.a1o); ot.aDe = xd(me.aDe); ot.aDo = xd(me.aDo);
        ot.aEnd = xd(me.aEnd); ot.vmax = xd(me.vmax); ot.jmax = xi(me.jmax); ot.bad = xi((int)me.bad) != 0;
        double tk, Fk;
        scan2::row_tF(rec_k(k), th0, lam, tk, Fk);
        scan2::out_join(h ? ot : me, h ? me : ot, tk, Fk, th0, lam, k, out);
    }
    __device__ __forceinline__ void out2(int lev, int Nl_, int k, double th0, double lam, const SolveOut& out, double* Xw) {
        const int qf = k, qb = Nl_ - 1 - k;
        const bool ok = !out.bad && out.zmax > 0.0 && out.zmax < 1e300;
        const double xk = h ? out.xkb : out.xkf;
        scan2::out_lane<true, false>(*this, lev, Nl_, h ? qb : qf, qf > qb ? qf : qb, h != 0, th0, lam, ok ? NORM_INFLATE / (xk * out.zmax) : 0.0,
                              -(h ? out.Ekb : out.Ekf), Xw);
    }
    __device__ __forceinline__ bool all(bool b) const { return __all_sync(FULL, b); }
    __device__ __forceinline__ bool any(bool b) const { return __any_sync(FULL, b); }
    __device__ __forceinline__ int min_i(int v) const { return __reduce_min_sync(FULL, v); }
    __device__ __forceinline__ int max_i(int v) const { return __reduce_max_sync(FULL, v); }
    __device__ __forceinline__ int first_i(int v) const {
        const unsigned m = __ballot_sync(FULL, v >= 0);
        return __shfl_sync(FULL, v, m ? (__ffs(m) - 1) : 0);
    }
    __device__ __forceinline__ void sync_mem() const { __syncwarp(); }
    __device__ __forceinline__ double ld(const double* p) const { return __ldcg(p); }
    // zero-fill invalid solves / form dX: one solve at a time (the forward lane of each flagged pair), rows dealt out over 32 lanes
    __device__ __forceinline__ void fixup(bool flag, double* Xrow, double* dXrow, int N_, bool bad, double hh, bool want_dX) {
        __syncwarp();
        unsigned m = __ballot_sync(FULL, flag) & 0xffffu;
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const bool bd = __shfl_sync(FULL, (int)bad, l) != 0;
            double* X = reinterpret_cast<double*>(__shfl_sync(FULL, reinterpret_cast<unsigned long long>(Xrow), l));
            double* dX = reinterpret_cast<double*>(__shfl_sync(FULL, reinterpret_cast<unsigned long long>(dXrow), l));
            fixup_solve(*this, X, want_dX ? dX : nullptr, N_, bd, hh, lane, 32);
        }
        __syncwarp();
    }
};

__global__ void __launch_bounds__(SC_WARPS * 32, IBS_SCAN2_CTAS)
scan2_solve_kernel(const ScanParams p) {
    extern __shared__ __align__(128) double sc_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, h = lane >> 4, li = lane & 15;
    Dev2Ctx ctx;
    ctx.ring = sc_smem + warp * S2_RING;
    ctx.bars = reinterpret_cast<uint64_t*>(sc_smem + SC_WARPS * S2_RING) + warp * SC_NSTAGE;
    // one block of cold state per PAIR of lanes (both run the same bookkeeping and store the same values)
    ColdState& cold = *reinterpret_cast<ColdState*>(sc_smem + SC_WARPS * S2_RING + SC_WARPS * SC_NSTAGE +
                                                    (size_t)(warp * scan2::NH + li) * COLD_STRIDE);
    ctx.parity = 0; ctx.lane = lane; ctx.h = h; ctx.N = p.N; ctx.warm = p.warm;
    if (lane == 0) {
        for (int s = 0; s < SC_NSTAGE; ++s) mbar_init(&ctx.bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const int N = p.N;
    for (;;) {
        int item = 0;
        if (lane == 0) item = (int)atomicAdd(p.counter, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= p.nitems) break;
        // Items are dealt in "column" order: round r holds the lines r, R + r, 2 R + r, ... (lc of them, all their theta0
        // groups), so that the previous LINE (line - 1: the adjacent alpha / surface of a scan grid, same theta0) was dealt
        // one whole round >= 2 x the resident warps earlier and has normally finished: its level eigenvalues are the warm
        // start (see the wait below).  The lines in flight
        // at any time are ~ resident warps / groups, as in plain line order (their records stay L2-resident).
        const int per_round = p.lc * p.groups;
        const int rnd = item / per_round, rem = item - rnd * per_round;
        const int jcol = rem / p.groups, grp = rem - jcol * p.groups;
        const int line = jcol * p.rounds + rnd;
        if (line >= p.nline) continue;
        const int slot = line * p.groups + grp;
        const int idx = grp * scan2::NH + li;
        const bool act = idx < p.nth0;
        const size_t sidx = (size_t)line * p.nth0 + (act ? idx : p.nth0 - 1);
        const double th0 = p.theta0[sidx];
        const double sg = p.sigma ? p.sigma[sidx] : 0.0;
        double* Xrow = (act && p.X_rows) ? p.X_rows + sidx * N : nullptr;
        double* dXrow = (act && p.dX_out) ? p.dX_out + sidx * N : nullptr;
        ItemProblem P;
        P.N = N; P.nlev = p.nlev; P.h = p.h; P.U = p.bounds[2 * line]; P.Lb = p.bounds[2 * line + 1];
        P.want_X = p.X_rows != nullptr; P.want_dX = p.dX_out != nullptr;
        P.safe = p.line_safe[line] != 0;
        ctx.line_base = p.poly + (size_t)line * p.rows_total * REC;
        int w_in = -1, w_out = -1;
        if (p.warm) {
            if (rnd > 0) {            // (lanes past nth0 duplicate the last theta0: so did the same lanes of the previous line)
                // The predecessor was dealt a whole round earlier and has normally finished; if not, wait for it: items are
                // claimed in order, so it is already running on a resident warp and waits only on still earlier items --
                // no deadlock -- and every line of rounds >= 1 is warm-started ALWAYS: the results do not depend on timing.
                if (lane == 0) {
                    const volatile unsigned* f = p.warm_flag + slot - p.groups;
                    unsigned spins = 0;
                    while (*f == 0u) {
                        __nanosleep(256);
                        if (++spins > (1u << 26)) __trap();              // a scheduling bug must trap, not hang the device
                    }
                }
                __syncwarp();
                __threadfence();
                w_in = ((slot - p.groups) * scan2::NH + li) * scan2::WREC;
            }
            if (rnd + 1 < p.rounds && line + 1 < p.nline) w_out = (slot * scan2::NH + li) * scan2::WREC;
        }
        ItemResult res;
        scan2::solve_item2(ctx, P, th0, act, sg, p.sigma != nullptr, Xrow, dXrow, res, cold, w_in, w_out);
        if (act && h == 0) {
            p.lam_out[sidx] = res.gam;
            if (p.lam_matrix_out) p.lam_matrix_out[sidx] = res.rho;
            if (p.info_out) p.info_out[sidx] = res.info;
        }
        // ---- publication of this item: its warm-start record (written inside solve_item2) and, for the fused arg-max (the
        // forward lanes carry the solves), its best (value, index) -- ONE fence for both (a fence
        // waits for the warp's outstanding stores, here the whole X output of the writing pass: ~2 % of the kernel each)
        const bool fused = p.items_per_surface > 0;
        const int surf = line / p.lines_per_surface;
        double bv = -INFINITY; int bi = 0x7fffffff, anynan = 0;
        if (fused) {
            if (act && h == 0) {
                const double v = res.gam;
                if (v != v) anynan = 1;
                best_merge(bv, bi, v, (line - surf * p.lines_per_surface) * p.nth0 + idx);
            }
            warp_best(bv, bi, anynan);
            if (lane == 0) {
                p.item_val[slot] = bv;
                p.item_idx[slot] = anynan ? -2 : bi;
            }
        }
        if (fused || w_out >= 0) {
            __threadfence();
            __syncwarp();
        }
        if (fused) {
            unsigned prev = 0;
            if (lane == 0) {
                if (w_out >= 0) *reinterpret_cast<volatile unsigned*>(p.warm_flag + slot) = 1u;
                prev = atomicAdd(&p.surf_count[surf], 1u);
            }
            surface_argmax_last(p, surf, prev, lane);
        } else if (w_out >= 0 && lane == 0) {
            *reinterpret_cast<volatile unsigned*>(p.warm_flag + slot) = 1u;
        }
    }
}

// ---- preparation: one CTA per field line ----------------------------------------------------------------
constexpr int PREP_T = 256;

template <class Op>
__device__ __forceinline__ double block_reduce(double v, Op op, double* scratch) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(FULL, v, o));
    __syncthreads();                                       // scratch free
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    double a = scratch[0];
    for (int w = 1; w < PREP_T / 32; ++w) a = op(a, scratch[w]);
    return a;
}
struct PMax { __device__ __forceinline__ double operator()(double a, double b) const { return fmax(a, b); } };
struct PMin { __device__ __forceinline__ double operator()(double a, double b) const { return fmin(a, b); } };

__global__ void __launch_bounds__(PREP_T)
scan_prep_kernel(const double* __restrict__ base, const double* __restrict__ dPdrho, const double* __restrict__ theta0, int nth0,
                 int N, double h2, int nlev, int rows_total, double* __restrict__ poly, double* __restrict__ bounds,
                 int* __restrict__ line_safe) {
    __shared__ double scratch[PREP_T / 32];
    const int line = blockIdx.x, tid = threadIdx.x;
    const double* b = base + (size_t)line * IBS_NBASE * N;
    const double dP = dPdrho[line];
    double t0 = 1e300, t1 = -1e300;
    for (int i = tid; i < nth0; i += PREP_T) { const double t = theta0[(size_t)line * nth0 + i]; t0 = fmin(t0, t); t1 = fmax(t1, t); }
    t0 = block_reduce(t0, PMin(), scratch);
    t1 = block_reduce(t1, PMax(), scratch);
    auto record = [&](int j) {
        return raw_record(b[(size_t)IBS_BASE_BMAG * N + j], b[(size_t)IBS_BASE_GRADPAR * N + j], b[(size_t)IBS_BASE_CVDRIFT * N + j],
                          b[(size_t)IBS_BASE_CVDRIFT0 * N + j], b[(size_t)IBS_BASE_GDS2 * N + j], b[(size_t)IBS_BASE_GDS21 * N + j],
                          b[(size_t)IBS_BASE_GDS22 * N + j], dP, h2);
    };
    double gmax = 0.0;
    for (int j = tid; j < N; j += PREP_T) {
        const Rec r = record(j);
        double gmn, gmx, cmn, cmx;
        record_ranges(r, t0, t1, gmn, gmx, cmn, cmx);
        if (gmx > gmax) gmax = gmx;
    }
    gmax = block_reduce(gmax, PMax(), scratch);
    const double sg = (gmax > 0.0 && gmax < 1e300) ? pow2(-exp_max2(gmax, 0.0)) : 1.0;
    double U = -1e300, minC = 1e300, maxg = 0.0, minF = 1e300, maxF = 0.0;
    double unsafe = 0.0;                                  // 1: some row could hold an invalid coefficient for some theta0 of the range
    double* out = poly + (size_t)line * rows_total * REC;
    for (int j = tid; j < N; j += PREP_T) {
        Rec r = record(j);
        r.G0 *= sg; r.G1 *= sg; r.G2 *= sg; r.C0 *= sg; r.C1 *= sg;
        double gmn, gmx, cmn, cmx;
        record_ranges(r, t0, t1, gmn, gmx, cmn, cmx);
        maxg = fmax(maxg, gmx);
        {
            // what the first output pass would test row by row (a = g + g' and F = g R positive and normal, C finite), certified
            // here for the whole theta0 range and all levels (R and C carry up to 4^MAXLEV there); NaN fails every comparison
            const double Fmn = gmn * r.R, Fmx = gmx * r.R;
            const bool ok = gmn >= 1e-290 && gmx <= 1e290 && Fmn >= 1e-290 && Fmx <= 1e290 && cmn >= -1e290 && cmx <= 1e290;
            if (!ok) unsafe = 1.0;
        }
        if (j >= 1 && j <= N - 2) {
            const double Fmin = gmn * r.R, Fmax = gmx * r.R;
            U = fmax(U, cmx >= 0.0 ? cmx / Fmin : cmx / Fmax);
            minC = fmin(minC, cmn); minF = fmin(minF, Fmin); maxF = fmax(maxF, Fmax);
        }
        int off = 0;
        for (int lev = 0; lev <= nlev; ++lev) {
            if (j & ((1 << lev) - 1)) break;
            const double f4 = (double)(1 << (2 * lev));
            double2* o = reinterpret_cast<double2*>(out + ((size_t)off + (j >> lev)) * REC);
            o[0] = make_double2(r.G0, r.G1);
            o[1] = make_double2(r.G2, r.C0 * f4);
            o[2] = make_double2(r.C1 * f4, r.R * f4);
            off += level_n(N, lev);
        }
    }
    U = block_reduce(U, PMax(), scratch);
    minC = block_reduce(minC, PMin(), scratch);
    maxg = block_reduce(maxg, PMax(), scratch);
    minF = block_reduce(minF, PMin(), scratch);
    maxF = block_reduce(maxF, PMax(), scratch);
    unsafe = block_reduce(unsafe, PMax(), scratch);
    if (tid == 0) {
        line_safe[line] = unsafe == 0.0 ? 1 : 0;
        U = U + 1e-12 * fabs(U) + 1e-300;
        const double numer = minC - 8.0 * maxg;
        bounds[2 * line + 0] = U;
        bounds[2 * line + 1] = 1.000001 * ((numer < 0.0) ? numer / minF : numer / maxF) - 1e-300;
    }
}

// ---- host side ---------------------------------------------------------------------------------------
bool scan_solver_eligible(const SolveParams& p) {
    if (const char* e = std::getenv("IBS_SCAN")) { if (std::atoi(e) == 0) return false; }
    if (p.line_of_solve || p.lam0 || p.g_out || p.c_out || p.f_out) return false;
    if (p.nth0 < 4 || (p.nsolve % p.nth0) != 0) return false;
    if ((p.N & 1) == 0 || p.N < 65) return false;          // composite Simpson by parity; matching-row margins
    return true;
}

// Launch of a lane kernel: persistent CTAs of SC_WARPS warps, as many as fit (IBS_MAX_CTAS_PER_SM caps the CTAs per SM) and
// no more than there are items for.  smem: the warps' record rings, their barriers and one cold-state block per solve.
template <void (*KERN)(ScanParams)>
static int lane_launch(const ScanParams& sp, size_t smem, cudaStream_t stream) {
    static bool configured[IBS_MAX_DEVICES] = {false};     // per kernel and per device (the attribute is per device)
    const int dslot = current_device_slot();
    if (!configured[dslot]) {
        IBS_CUDA_CHECK(cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        IBS_CUDA_CHECK(cudaFuncSetAttribute(KERN, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        configured[dslot] = true;
    }
    int per_sm = 0;
    IBS_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, KERN, SC_WARPS * 32, smem));
    if (per_sm < 1) per_sm = 1;
    if (const char* e = std::getenv("IBS_MAX_CTAS_PER_SM")) { const int v = std::atoi(e); if (v >= 1 && v < per_sm) per_sm = v; }
    const long long cap = (long long)num_sms() * per_sm;
    const long long need = ((long long)sp.nitems + SC_WARPS - 1) / SC_WARPS;
    const int grid = (int)(need < cap ? need : cap);
    KERN<<<grid, SC_WARPS * 32, smem, stream>>>(sp);
    IBS_CUDA_CHECK(cudaGetLastError());
    return IBS_OK;
}
// which of the two lane kernels a batch of N-point lines goes to (IBS_SCAN2=0: always the two-chains-per-lane kernel)
static bool use_scan2(int N) {
    if (const char* e = std::getenv("IBS_SCAN2")) { if (std::atoi(e) == 0) return false; }
    return scan2::scan2_size_ok(N);
}

// One launch set (prep + solver) for the lines [l0, l0 + nline) of the batch p
static int scan_solve_lines(const SolveParams& p, int l0, int nline, cudaStream_t stream) {
    const int N = p.N;
    const int nlev = num_levels(N);
    const int rows_total = level_offset(N, nlev + 1);
    const size_t v0 = (size_t)l0 * p.nth0, nsolve = (size_t)nline * p.nth0;
    const bool s2 = use_scan2(N);
    const int groups = s2 ? (p.nth0 + scan2::NH - 1) / scan2::NH : (p.nth0 + 31) / 32;
    const int nitems = nline * groups;
    const bool fused = p.lines_per_surface > 0 && p.best_out;
    const int nsurf = fused ? nline / p.lines_per_surface : 0;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_poly = take((size_t)nline * rows_total * REC * sizeof(double));
    const size_t o_bounds = take((size_t)nline * 2 * sizeof(double));
    const size_t o_safe = take((size_t)nline * sizeof(int));
    // lane-per-chain kernel: column order of the lines + warm start from the previous line (see scan2_solve_kernel); a round
    // is at least IBS_SCAN_WARM_SPACING (default 2) x the resident warps, so that a line's predecessor has normally finished
    int lc = nline, rounds = 1;
    bool warm = s2;
    if (const char* e = std::getenv("IBS_SCAN_WARM")) { if (std::atoi(e) == 0) warm = false; }
    if ((long long)nitems * scan2::NH * scan2::WREC > 0x7fffffffLL) warm = false;           // (tokens are int element offsets)
    if (warm) {
        // Measured (D3D config x 37 equilibria, B200): a round of 1.0 / 1.25 / 1.5 / 2.0 / 3.0 x the resident warps -> solver
        // 3.49 / 3.26 / 3.22 / 3.04 / 3.08 ms (no warm start: 3.47): closer rounds wait on their predecessors, wider ones
        // leave a larger cold first round.
        double spacing = 2.0;
        if (const char* e = std::getenv("IBS_SCAN_WARM_SPACING")) { const double v = std::atof(e); if (v >= 1.0 && v <= 16.0) spacing = v; }
        const long long resident = (long long)num_sms() * IBS_SCAN2_CTAS * SC_WARPS;
        const long long lc0 = (long long)std::ceil(spacing * (double)resident / groups);       // lines per round, at least
        rounds = (int)(nline / lc0);
        if (rounds >= 2) lc = (nline + rounds - 1) / rounds;                                    // (>= lc0)
        else rounds = 1;
        if (rounds < 2) warm = false;
    }
    const size_t nzero = 1 + (size_t)nsurf + (warm ? (size_t)nitems : 0);
    const size_t o_zero = take(nzero * sizeof(unsigned));             // work counter + per-surface counters + warm-start flags: zeroed together
    const size_t o_warm = take(warm ? (size_t)nitems * scan2::NH * scan2::WREC * sizeof(double) : 0);
    const size_t o_ival = take(fused ? (size_t)nitems * sizeof(double) : 0);
    const size_t o_iidx = take(fused ? (size_t)nitems * sizeof(int) : 0);
    const size_t xs_bytes = (p.dX_out && !p.X_out) ? nsolve * N * sizeof(double) : 0;      // X is the scratch dX is formed from
    const size_t o_xs = take(xs_bytes);
    char* ws = nullptr;
    IBS_CUDA_CHECK(cudaMallocAsync((void**)&ws, off + 256, stream));
    int rc = IBS_OK;
    ScanParams sp;
    sp.poly = (double*)(ws + o_poly); sp.bounds = (double*)(ws + o_bounds); sp.line_safe = (int*)(ws + o_safe); sp.counter = (unsigned*)(ws + o_zero);
    sp.theta0 = p.theta0 + v0; sp.sigma = p.sigma ? p.sigma + v0 : nullptr;
    sp.nline = nline; sp.nth0 = p.nth0; sp.N = N; sp.nlev = nlev; sp.rows_total = rows_total;
    sp.groups = groups;
    sp.lc = lc; sp.rounds = rounds;
    sp.nitems = s2 ? rounds * lc * groups : nitems;          // (column order: padded; slots past nline are skipped)
    sp.h = p.h;
    sp.lam_out = p.lam_out + v0;
    sp.lam_matrix_out = p.lam_matrix_out ? p.lam_matrix_out + v0 : nullptr;
    sp.X_out = p.X_out ? p.X_out + v0 * N : nullptr;
    sp.dX_out = p.dX_out ? p.dX_out + v0 * N : nullptr;
    sp.info_out = p.info_out ? p.info_out + v0 : nullptr;
    sp.X_rows = sp.X_out ? sp.X_out : (xs_bytes ? (double*)(ws + o_xs) : nullptr);
    sp.items_per_surface = fused ? p.lines_per_surface * groups : 0;
    sp.lines_per_surface = fused ? p.lines_per_surface : 1;
    sp.item_val = (double*)(ws + o_ival); sp.item_idx = (int*)(ws + o_iidx);
    sp.surf_count = sp.counter + 1;
    sp.warm = warm ? (double*)(ws + o_warm) : nullptr;
    sp.warm_flag = warm ? sp.counter + 1 + nsurf : nullptr;
    const size_t surf0 = fused ? (size_t)l0 / p.lines_per_surface : 0;
    sp.best_out = fused ? p.best_out + 2 * surf0 : nullptr;
    sp.sigma0_out = (fused && p.sigma0_out) ? p.sigma0_out + surf0 : nullptr;
    if (cudaError_t e = cudaMemsetAsync(sp.counter, 0, nzero * sizeof(unsigned), stream); e != cudaSuccess)
        rc = cuda_fail(e, "cudaMemsetAsync(scan counters)");
    if (rc == IBS_OK) {
        scan_prep_kernel<<<nline, PREP_T, 0, stream>>>(p.base + (size_t)l0 * IBS_NBASE * N, p.dPdrho + l0, sp.theta0, p.nth0, N, p.h * p.h, nlev,
                                                       rows_total, (double*)(ws + o_poly), (double*)(ws + o_bounds), (int*)(ws + o_safe));
        if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) rc = cuda_fail(e, "scan_prep_kernel launch");
    }
    if (rc == IBS_OK) {
        const size_t ring_bars = (size_t)SC_WARPS * SC_NSTAGE * sizeof(uint64_t);
        if (s2)        // one cold-state block per pair of lanes
            rc = lane_launch<scan2_solve_kernel>(sp, (size_t)SC_WARPS * S2_RING * sizeof(double) + ring_bars +
                                                         (size_t)SC_WARPS * scan2::NH * COLD_STRIDE * sizeof(double), stream);
        else
            rc = lane_launch<scan_solve_kernel>(sp, (size_t)SC_WARPS * SC_RING * sizeof(double) + ring_bars +
                                                        (size_t)SC_WARPS * 32 * COLD_STRIDE * sizeof(double), stream);
    }
    cudaFreeAsync(ws, stream);
    return rc;
}

int scan_solve_dispatch(const SolveParams& p, cudaStream_t stream) {
    const int nline = p.nsolve / p.nth0;
    keep_pool_cached();
    // The coefficient records take ~95 KB per field line (N = 1025): very large batches are processed in chunks of lines so
    // that the stream-ordered workspace stays below IBS_SCAN_WS_MB (default 8 GB; the chunks are still >> one round of warps).
    size_t ws_mb = 8192;
    if (const char* e = std::getenv("IBS_SCAN_WS_MB")) { const long v = std::atol(e); if (v >= 1) ws_mb = (size_t)v; }
    const size_t per_line = (size_t)level_offset(p.N, num_levels(p.N) + 1) * REC * sizeof(double) + 64;
    long long chunk = (long long)((ws_mb << 20) / per_line);
    if (chunk < 1) chunk = 1;
    if (p.lines_per_surface > 0 && p.best_out) {           // fused arg-max: a chunk holds whole surfaces
        IBS_REQUIRE(nline % p.lines_per_surface == 0, "nline must be a multiple of lines_per_surface");
        chunk = (chunk / p.lines_per_surface) * p.lines_per_surface;
        if (chunk < p.lines_per_surface) chunk = p.lines_per_surface;
    }
    int rc = IBS_OK;
    for (long long l0 = 0; l0 < nline && rc == IBS_OK; l0 += chunk)
        rc = scan_solve_lines(p, (int)l0, (int)((nline - l0 < chunk) ? (nline - l0) : chunk), stream);
    return rc;
}

}  // namespace ibs
