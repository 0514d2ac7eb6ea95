// kernel_lead.cuh — shared-memory slab kernel for backorder lead-time models
// (LeadtimeRecursion.java:49-73 with the lambdas of Leadtime.java:50-81; lead time 1, and the lead
// time 2 extension of config C4).  Brute force per real state, bit-identical to bi_generic.
//
// State (x, q1[, q2]); stock level l = x + q1 - d; successor (succ(l), [q2,] a).  For a fixed action a
// (and column q2) the successor values V_{t+1}[succ(y - d_j), q2, a] of consecutive levels
// y = x + q1 slide by one row per demand step, exactly like the 1-D kernel — so a thread owns one
// action a, YT = 4 consecutive preQ1 (levels) and RQ preQ2 columns, i.e. 4*RQ states:
//   per demand point it loads ONE new row of RQ values and one level cost from shared memory, forms
//   cst = fv_a + L(level) once, m_k = p*cst_k for its 4 levels (shared by the RQ columns), and then
//   spends (mul, add, add) on each evaluation: (1 + 4 + 3*4*RQ) / (4*RQ) = 3.31 fp64 instr per eval
//   for RQ = 4 (5 in bi_backorder_staged), and 3.5 B of shared memory per eval instead of 8 B of L1.
// A CTA takes one inventory level x, NYB = 4*NYT consecutive preQ1, RQ consecutive preQ2 and all
// actions; the slab of successor rows it can reach, slab[level window][RQ][A], is staged once
// (coalesced along a).  Q-values go back through shared memory (aliasing the slab) for the
// lexicographic (value, action) argopt per state.  Needs consecutive integer demands and a slab
// that fits in shared memory; otherwise bi_backorder_staged runs.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>

#include "dev_model.cuh"
#include "kernel_tiled.cuh"  // lds_double2

namespace sdpb {

constexpr int kLeadYT = 4;

struct LeadArgs {
    int t, D, pmf_off;
    const double* Vn;
    double* Vt;
    int* Qt;
    long long lo, hi;
    long long row0;      // first inventory row (or virtual level tile origin) of the range
    int NYT;             // level groups per CTA (NYB = 4 * NYT levels)
    int ny_tiles, nq2_tiles;
    int A, Apad, di_max, NR;  // actions, padded row length, max demand index, slab rows
    int nthreads;
};

__device__ __forceinline__ long long lds_s64(unsigned shared_addr) {
    long long v;
    asm volatile("ld.shared.s64 %0, [%1];" : "=l"(v) : "r"(shared_addr));
    return v;
}

// one fp64 value at base + byte offset, through the read-only path
__device__ __forceinline__ double ldg_at(const char* base, long long byte_off) {
    return __ldg(reinterpret_cast<const double*>(base + byte_off));
}

__device__ __forceinline__ double lds_double(unsigned shared_addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(shared_addr));
    return v;
}

template <bool IS_MIN, bool LAST, int RQ, bool DEDUP>
__global__ void __launch_bounds__(256)
bi_lead_slab(const __grid_constant__ DevModel M, const __grid_constant__ LeadArgs a) {
    constexpr int YT = kLeadYT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NYB = YT * a.NYT;
    const int D = a.D, A = a.A, Apad = a.Apad;
    // layout: [ slab NR*RQ*Apad doubles | later: Q-values NYB*RQ*Apad ] [ Lw NR doubles ] [ PP D double2 ]
    double* slab = reinterpret_cast<double*>(smem_raw);
    const size_t slab_elems = (size_t)max(a.NR, NYB) * RQ * Apad;
    double* Lw = slab + slab_elems;
    double2* PP = reinterpret_cast<double2*>(Lw + ((a.NR + 1) & ~1));

    // ---- which states: one x (or none when folded), NYB consecutive levels, RQ consecutive preQ2 ----
    long long b = blockIdx.x;
    int q2_0 = 0;
    if (M.lead == 2) { q2_0 = (int)(b % a.nq2_tiles) * RQ; b /= a.nq2_tiles; }
    const int ytile = (int)(b % a.ny_tiles); b /= a.ny_tiles;
    // real grid: level y = ix + q1 with q1 = ytile*NYB + local; folded grid: level = ytile*NYB + local
    const long long ix = DEDUP ? 0 : a.row0 + b;
    const int q1_0 = ytile * NYB;
    const long long y0 = ix + q1_0;  // level index of local 0
    const int n_levels = DEDUP ? (M.nI + M.nQ - 1) : M.nQ;  // valid range of (q1_0 + local)

    const int tid = threadIdx.x;
    for (int j = tid; j < D; j += a.nthreads) PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
    const bool lost = (M.flags & SDPB_F_LOST_SALES) != 0;
    const long long strideX = (M.lead == 2) ? (long long)M.nQ * M.nQ : (long long)M.nQ;
    // window index wi <-> unclamped level index il = y0 - di_max + wi
    for (int wi = tid; wi < a.NR; wi += a.nthreads) {
        const double lvl = M.inv_min + (double)(y0 - a.di_max + wi) * M.step;
        Lw[wi] = M.h * fmax(lvl, 0.0) + M.pen * fmax(-lvl, 0.0);
    }
    if (!LAST) {
        // one warp per (window row, column block): coalesced along the action, no integer division
        const int warp_s = tid >> 5, lane_s = tid & 31, nwarps_s = a.nthreads >> 5;
        for (int row = warp_s; row < a.NR * RQ; row += nwarps_s) {
            const int wi = row / RQ, rr = row - wi * RQ;  // RQ is a compile-time constant
            long long is = y0 - a.di_max + wi;
            if (lost) is = is > M.i_zero ? is : M.i_zero;
            is = is < M.nI - 1 ? is : M.nI - 1;  // upper clamp first; also the memory-safety clip
            is = is > 0 ? is : 0;
            const int q2 = min(q2_0 + rr, M.nQ - 1);
            const double* __restrict__ src = a.Vn + is * strideX + ((M.lead == 2) ? (long long)q2 * M.nQ : 0);
            // asynchronous 8-byte copies (LDGSTS): every load of the slab is in flight before any is
            // waited for, so staging costs one memory latency instead of one per row
            const unsigned dst = (unsigned)__cvta_generic_to_shared(slab + (size_t)row * Apad);
            for (int ai = lane_s; ai < A; ai += 32)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + (unsigned)ai * 8u), "l"(src + ai));
        }
        asm volatile("cp.async.commit_group;");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();

    const int g = tid / A, ai = tid - g * A;  // level group, action
    const bool worker = g < a.NYT;
    double acc[YT][RQ];
#pragma unroll
    for (int k = 0; k < YT; k++)
#pragma unroll
        for (int r = 0; r < RQ; r++) acc[k][r] = 0.0;

    if (worker) {
        const double av = (double)ai * M.step;
        const double fv = (av > 0.0 ? M.K : 0.0) + M.v_t[a.t - 1] * av;  // Leadtime.java:73-74,79
        const unsigned slab_s = (unsigned)__cvta_generic_to_shared(slab) + (unsigned)ai * 8u;
        const unsigned lw_s = (unsigned)__cvta_generic_to_shared(Lw);
        const unsigned pp_s = (unsigned)__cvta_generic_to_shared(PP);
        const unsigned row_bytes = (unsigned)(RQ * Apad) * 8u;
        // level slot k at demand j needs window row  wi = 4g + k + (D-1-j)
        int wi0 = YT * g + (D - 1);
        double cst[YT], Vw[YT][RQ];
#pragma unroll
        for (int k = 0; k < YT; k++) {
            cst[k] = fv + lds_double(lw_s + (unsigned)(wi0 + k) * 8u);
#pragma unroll
            for (int r = 0; r < RQ; r++)
                Vw[k][r] = LAST ? 0.0 : lds_double(slab_s + (unsigned)(wi0 + k) * row_bytes + (unsigned)(r * Apad) * 8u);
        }
#define SDPB_LEAD_STEP(JJ)                                                                          \
        {                                                                                               \
            const double2 pp = lds_double2(pp_s + (unsigned)j * 16u);                                   \
            const int wn = max(wi0 - 1, 0);                                                             \
            const double lnew = lds_double(lw_s + (unsigned)wn * 8u);                                   \
            double vnew[RQ];                                                                            \
            _Pragma("unroll") for (int r = 0; r < RQ; r++)                                              \
                vnew[r] = LAST ? 0.0 : lds_double(slab_s + (unsigned)wn * row_bytes + (unsigned)(r * Apad) * 8u); \
            _Pragma("unroll") for (int k = 0; k < YT; k++) {                                            \
                const int ph = (k - (JJ)) & 3;                                                          \
                const double m = pp.x * cst[ph];                    /* p_j * c(s,a,d_j) */            \
                _Pragma("unroll") for (int r = 0; r < RQ; r++) {                                        \
                    acc[k][r] += m;                                 /* LeadtimeRecursion.java:59 */    \
                    if (!LAST) acc[k][r] += pp.y * Vw[ph][r];       /* LeadtimeRecursion.java:62 */    \
                }                                                                                       \
            }                                                                                           \
            const int pn = (3 - (JJ)) & 3;                                                              \
            cst[pn] = fv + lnew;                                                                        \
            _Pragma("unroll") for (int r = 0; r < RQ; r++) Vw[pn][r] = vnew[r];                         \
            wi0 -= 1;                                                                                   \
            j += 1;                                                                                     \
        }
        int j = 0;
        for (; j + 4 <= D;) { SDPB_LEAD_STEP(0) SDPB_LEAD_STEP(1) SDPB_LEAD_STEP(2) SDPB_LEAD_STEP(3) }
        if (j < D) SDPB_LEAD_STEP(0)
        if (j < D) SDPB_LEAD_STEP(1)
        if (j < D) SDPB_LEAD_STEP(2)
#undef SDPB_LEAD_STEP
    }

    // ---- Q-values to shared memory (aliasing the slab), then one warp per state picks the optimum ----
    __syncthreads();
    double* Qs = slab;  // [NYB][RQ][Apad]
    if (worker) {
#pragma unroll
        for (int k = 0; k < YT; k++)
#pragma unroll
            for (int r = 0; r < RQ; r++) Qs[((size_t)(YT * g + k) * RQ + r) * Apad + ai] = acc[k][r];
    }
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31, nwarps = a.nthreads >> 5;
    for (int s = warp; s < NYB * RQ; s += nwarps) {
        const int local = s / RQ, r = s - local * RQ;
        const double* q = Qs + (size_t)s * Apad;
        double best = IS_MIN ? DBL_MAX : -DBL_MAX;
        int besti = kNoAction;
        for (int i = lane; i < A; i += 32) {  // ascending within a lane: first optimum wins
            const double v = q[i];
            if (IS_MIN ? (v < best) : (v > best)) { best = v; besti = i; }
        }
#pragma unroll
        for (int sh = 16; sh > 0; sh >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, sh);
            const int oi = __shfl_xor_sync(0xffffffffu, besti, sh);
            if (better<IS_MIN>(ov, oi, best, besti)) { best = ov; besti = oi; }
        }
        if (lane == 0) {
            const int lev = q1_0 + local;
            const int q2 = q2_0 + r;
            if (lev < n_levels && (M.lead != 2 || q2 < M.nQ)) {
                long long idx = DEDUP ? (long long)lev : ix * M.nQ + lev;
                if (M.lead == 2) idx = idx * M.nQ + q2;
                if (idx >= a.lo && idx < a.hi) {
                    a.Vt[idx] = best;
                    a.Qt[idx] = besti == kNoAction ? -1 : besti;
                }
            }
        }
    }
}

// ---- host side --------------------------------------------------------------------------------
struct LeadPlan {
    bool ok = false;
    int NYT = 0, RQ = 1, Apad = 0, nthreads = 0, di_max = 0, span = 0, NR = 0;
    size_t smem = 0;
};

// Plan for one period; ok == false means "use bi_backorder_staged".
inline LeadPlan plan_lead(const sdpb_model& m, const DevModel& d, int D, const int* di) {
    LeadPlan P;
    if (m.cost_kind != SDPB_COST_BACKORDER || m.lead_time < 1) return P;
    int lo = di[0], hi = di[0];
    for (int j = 0; j < D; j++) {
        if (di[j] != di[0] + j) return P;  // the register window needs consecutive demands
        lo = std::min(lo, di[j]);
        hi = std::max(hi, di[j]);
    }
    const int A = d.max_order_idx + 1;
    P.RQ = m.lead_time == 2 ? 4 : 1;
    P.NYT = std::max(1, std::min(256 / A, 4));
    if (A > 256) return P;
    P.Apad = (A + 1) & ~1;
    P.nthreads = std::min(256, ((P.NYT * A + 31) / 32) * 32);
    P.di_max = hi;
    P.span = hi - lo;
    const int NYB = kLeadYT * P.NYT;
    P.NR = NYB + P.span;
    P.smem = ((size_t)std::max(P.NR, NYB) * P.RQ * P.Apad + ((P.NR + 1) & ~1)) * 8 + (size_t)D * 16 + 16;
    P.ok = P.smem <= 110 * 1024;  // two CTAs per SM
    return P;
}

template <bool DEDUP>
inline int launch_lead(const LeadPlan& P, const DevModel& dm, int t, int D, int pmf_off, const double* Vn,
                       double* Vt, int* Qt, long long lo, long long hi, cudaStream_t stream) {
    if (hi <= lo) return SDPB_OK;
    LeadArgs a;
    a.t = t; a.D = D; a.pmf_off = pmf_off; a.Vn = Vn; a.Vt = Vt; a.Qt = Qt; a.lo = lo; a.hi = hi;
    a.NYT = P.NYT; a.A = dm.max_order_idx + 1; a.Apad = P.Apad; a.di_max = P.di_max; a.NR = P.NR;
    a.nthreads = P.nthreads;
    const int NYB = kLeadYT * P.NYT;
    a.nq2_tiles = dm.lead == 2 ? (dm.nQ + P.RQ - 1) / P.RQ : 1;
    long long rows;
    if (DEDUP) {
        a.ny_tiles = (dm.nI + dm.nQ - 1 + NYB - 1) / NYB;
        a.row0 = 0;
        rows = 1;
    } else {
        a.ny_tiles = (dm.nQ + NYB - 1) / NYB;
        const long long per_x = dm.lead == 2 ? (long long)dm.nQ * dm.nQ : (long long)dm.nQ;
        a.row0 = lo / per_x;
        rows = (hi - 1) / per_x - a.row0 + 1;
    }
    const long long blocks = rows * a.ny_tiles * a.nq2_tiles;
    const bool last = (Vn == nullptr), mn = dm.is_min != 0;  // period T without a terminal table
    cudaError_t e = cudaSuccess;
#define SDPB_LEAD_LAUNCH(MN, LS, RQ_)                                                                  \
    {                                                                                                  \
        auto k = bi_lead_slab<MN, LS, RQ_, DEDUP>;                                                     \
        if (P.smem > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.smem); \
        if (e == cudaSuccess) k<<<(unsigned)blocks, P.nthreads, P.smem, stream>>>(dm, a);              \
    }
    if (P.RQ == 4) {
        if (mn) { if (last) SDPB_LEAD_LAUNCH(true, true, 4) else SDPB_LEAD_LAUNCH(true, false, 4) }
        else    { if (last) SDPB_LEAD_LAUNCH(false, true, 4) else SDPB_LEAD_LAUNCH(false, false, 4) }
    } else {
        if (mn) { if (last) SDPB_LEAD_LAUNCH(true, true, 1) else SDPB_LEAD_LAUNCH(true, false, 1) }
        else    { if (last) SDPB_LEAD_LAUNCH(false, true, 1) else SDPB_LEAD_LAUNCH(false, false, 1) }
    }
#undef SDPB_LEAD_LAUNCH
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    return SDPB_OK;
}

// ---------------------------------------------------------------------------------------------
// bi_lead_col — one thread per successor COLUMN.  For a fixed inventory level x and a fixed column
// c = (preQ2, a) the values G(y, c), y = x + preQ1, form a 1-D sliding problem along preQ1 with the
// column's own value vector V_{t+1}[., c]: the row slot k needs at demand j+1 is the row slot k-1
// needed at demand j.  So a thread walks the whole preQ1 axis in chunks of YT = 8 levels, keeps the 8
// level costs and 8 successor values in registers (rotation unrolled x8), and per demand point loads
// ONE new value of its column straight from global memory (lanes = consecutive columns: coalesced;
// every row is re-read D/8 times by the same thread, so L1 serves it) and one level cost from shared
// memory (CTA-uniform: a broadcast).  fp64 per evaluation: (1 + 8 + 8 + 16) / 8 = 4.125; no slab
// staging, no per-tile set-up.  A CTA is NQB whole preQ2 values x all actions (505 of 512 threads
// busy for C4), so the argopt over a stays inside the CTA: after each chunk the 8 x NQB states are
// reduced through shared memory with the lexicographic (value, action) rule.
constexpr int kColYT = 8;  // levels per chunk

struct ColArgs {
    int t, D, pmf_off;
    const double* Vn;
    double* Vt;
    int* Qt;
    long long lo, hi;
    long long row0;           // first inventory row of the range (real grid)
    int A, NQB, nq2_groups;   // actions; preQ2 values per CTA; CTAs along preQ2
    int LT, n_ltiles;         // levels (preQ1 values) per CTA (multiple of 8), CTAs along the level axis
    int di_max, NRW;          // window rows = LT + span
    int nthreads;
};

template <bool IS_MIN, bool LAST, bool DEDUP>
__global__ void __launch_bounds__(512, 1)
bi_lead_col(const __grid_constant__ DevModel M, const __grid_constant__ ColArgs a) {
    constexpr int YT = kColYT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.D, A = a.A;
    // layout: [ red 2 x YT*nthreads doubles (double-buffered) ][ Lw NRW doubles ][ RO NRW int64 row offsets ][ PP D double2 ]
    double* red_base = reinterpret_cast<double*>(smem_raw);
    double* Lw = red_base + (size_t)2 * YT * a.nthreads;
    long long* RO = reinterpret_cast<long long*>(Lw + a.NRW);
    double2* PP = reinterpret_cast<double2*>(smem_raw + ((((size_t)2 * YT * a.nthreads + 2 * (size_t)a.NRW) * 8 + 15) & ~(size_t)15));

    long long b = blockIdx.x;
    const int q2g = (int)(b % a.nq2_groups); b /= a.nq2_groups;
    const int lt = (int)(b % a.n_ltiles); b /= a.n_ltiles;
    const long long ix = DEDUP ? 0 : a.row0 + b;
    const int l_begin = lt * a.LT;
    const int n_levels = DEDUP ? (M.nI + M.nQ - 1) : M.nQ;
    const int l_end = min(l_begin + a.LT, n_levels);
    const long long y_tile0 = ix + l_begin;  // level index of the tile's first level

    const int tid = threadIdx.x;
    const int qq = tid / A, ai = tid - qq * A;
    const int q2 = q2g * a.NQB + qq;
    const bool worker = qq < a.NQB && (M.lead != 2 || q2 < M.nQ);
    const bool lost = (M.flags & SDPB_F_LOST_SALES) != 0;
    const long long strideX = (M.lead == 2) ? (long long)M.nQ * M.nQ : (long long)M.nQ;

    for (int j = tid; j < D; j += a.nthreads) PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
    // window index wi <-> unclamped level index il = y_tile0 - di_max + wi
    for (int wi = tid; wi < a.NRW; wi += a.nthreads) {
        const long long il = y_tile0 - a.di_max + wi;
        const double lvl = M.inv_min + (double)il * M.step;
        Lw[wi] = M.h * fmax(lvl, 0.0) + M.pen * fmax(-lvl, 0.0);
        long long is = il;
        if (lost) is = is > M.i_zero ? is : M.i_zero;
        is = is < M.nI - 1 ? is : M.nI - 1;  // upper clamp first; also the memory-safety clip
        is = is > 0 ? is : 0;
        RO[wi] = is * strideX * (long long)sizeof(double);  // byte offset of the successor's row
    }
    __syncthreads();

    const double av = (double)ai * M.step;
    const double fv = (av > 0.0 ? M.K : 0.0) + M.v_t[a.t - 1] * av;  // Leadtime.java:73-74,79
    const char* __restrict__ col = reinterpret_cast<const char*>(
        a.Vn + ((M.lead == 2) ? (long long)min(q2, M.nQ - 1) * M.nQ + ai : (long long)ai));
    const unsigned lw_s = (unsigned)__cvta_generic_to_shared(Lw);
    const unsigned ro_s = (unsigned)__cvta_generic_to_shared(RO);
    const unsigned pp_s = (unsigned)__cvta_generic_to_shared(PP);
    const int warp = tid >> 5, lane = tid & 31, nwarps = a.nthreads >> 5;

    int parity = 0;
    for (int l0 = l_begin; l0 < l_end; l0 += YT, parity ^= 1) {
        // Q-values of this chunk go to buffer `parity`; the other buffer may still be read by slower
        // warps finishing the previous chunk's argopt, so one barrier per chunk is enough.
        double* red_v = red_base + (size_t)parity * YT * a.nthreads;
        double acc[YT], cst[YT], Vw[YT];
#pragma unroll
        for (int k = 0; k < YT; k++) acc[k] = 0.0;
        if (worker) {
            // level slot k at demand j needs window row  wi = (l0 - l_begin) + k + (D-1-j)
            int wi0 = (l0 - l_begin) + (D - 1);
#pragma unroll
            for (int k = 0; k < YT; k++) {
                const int wi = min(wi0 + k, a.NRW - 1);
                cst[k] = fv + lds_double(lw_s + (unsigned)wi * 8u);
                Vw[k] = LAST ? 0.0 : ldg_at(col, lds_s64(ro_s + (unsigned)wi * 8u));
            }
            // two-deep software pipeline on the global loads: `pre` is the value entering at step j+1
            double pre = 0.0;
            if (!LAST) pre = ldg_at(col, lds_s64(ro_s + (unsigned)max(wi0 - 1, 0) * 8u));
#define SDPB_COL_STEP(JJ)                                                                             \
            {                                                                                             \
                const double2 pp = lds_double2(pp_s + (unsigned)j * 16u);                                 \
                const double vnew = pre;                                                                  \
                if (!LAST) pre = ldg_at(col, lds_s64(ro_s + (unsigned)max(wi0 - 2, 0) * 8u));             \
                const double lnew = lds_double(lw_s + (unsigned)max(wi0 - 1, 0) * 8u);                    \
                _Pragma("unroll") for (int k = 0; k < YT; k++) {                                          \
                    const int ph = (k - (JJ)) & (YT - 1);                                                 \
                    acc[k] += pp.x * cst[ph];                      /* LeadtimeRecursion.java:59 */       \
                    if (!LAST) acc[k] += pp.y * Vw[ph];            /* LeadtimeRecursion.java:62 */       \
                }                                                                                         \
                const int pn = (YT - 1 - (JJ)) & (YT - 1);                                                \
                cst[pn] = fv + lnew;                                                                      \
                Vw[pn] = vnew;                                                                            \
                wi0 -= 1;                                                                                 \
                j += 1;                                                                                   \
            }
            int j = 0;
            for (; j + YT <= D;) {
#pragma unroll
                for (int jj = 0; jj < YT; jj++) SDPB_COL_STEP(jj)
            }
#pragma unroll
            for (int jj = 0; jj < YT - 1; jj++)
                if (j < D) SDPB_COL_STEP(jj)
#undef SDPB_COL_STEP
        }
        // ---- argopt over the actions of each of the YT x NQB states of this chunk ----
#pragma unroll
        for (int k = 0; k < YT; k++) red_v[(size_t)k * a.nthreads + tid] = acc[k];
        __syncthreads();
        for (int s = warp; s < YT * a.NQB; s += nwarps) {
            const int k = s / a.NQB, sq = s - k * a.NQB;
            const double* q = red_v + (size_t)k * a.nthreads + sq * A;
            double best = IS_MIN ? DBL_MAX : -DBL_MAX;
            int besti = kNoAction;
            for (int i = lane; i < A; i += 32) {  // ascending within a lane: first optimum wins
                const double v = q[i];
                if (IS_MIN ? (v < best) : (v > best)) { best = v; besti = i; }
            }
#pragma unroll
            for (int sh = 16; sh > 0; sh >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, best, sh);
                const int oi = __shfl_xor_sync(0xffffffffu, besti, sh);
                if (better<IS_MIN>(ov, oi, best, besti)) { best = ov; besti = oi; }
            }
            if (lane == 0) {
                const int lev = l0 + k;
                const int sq2 = q2g * a.NQB + sq;
                if (lev < l_end && (M.lead != 2 || sq2 < M.nQ)) {
                    long long idx = DEDUP ? (long long)lev : ix * M.nQ + lev;
                    if (M.lead == 2) idx = idx * M.nQ + sq2;
                    if (idx >= a.lo && idx < a.hi) {
                        a.Vt[idx] = best;
                        a.Qt[idx] = besti == kNoAction ? -1 : besti;
                    }
                }
            }
        }
    }
}

struct ColPlan {
    bool ok = false;
    int NQB = 1, nthreads = 0, LT = 0, di_max = 0, span = 0, NRW = 0;
    size_t smem = 0;
};

inline ColPlan plan_col(const sdpb_model& m, const DevModel& d, int D, const int* di, bool dedup) {
    ColPlan P;
    if (m.cost_kind != SDPB_COST_BACKORDER || m.lead_time < 1) return P;
    int lo = di[0], hi = di[0];
    for (int j = 0; j < D; j++) {
        if (di[j] != di[0] + j) return P;  // the register window needs consecutive demands
        lo = std::min(lo, di[j]);
        hi = std::max(hi, di[j]);
    }
    const int A = d.max_order_idx + 1;
    if (A > 512) return P;
    const int max_threads = 512;  // measured best on C4 (512: 238 ms, 128: 244, 224: 270, 320: 317)
    P.NQB = m.lead_time == 2 ? std::max(1, std::min(max_threads / A, d.nQ)) : 1;
    P.nthreads = ((P.NQB * A + 31) / 32) * 32;
    const int n_levels = dedup ? d.nI + d.nQ - 1 : d.nQ;
    // real grid: one CTA walks the whole preQ1 axis; folded grid: 64 levels per CTA for parallelism
    P.LT = dedup ? 64 : ((n_levels + kColYT - 1) / kColYT) * kColYT;
    P.di_max = hi;
    P.span = hi - lo;
    P.NRW = P.LT + P.span;
    P.smem = ((((size_t)2 * kColYT * P.nthreads + 2 * (size_t)P.NRW) * 8 + 15) & ~(size_t)15) + (size_t)D * 16 + 16;
    P.ok = P.smem <= 100 * 1024;
    return P;
}

template <bool DEDUP>
inline int launch_col(const ColPlan& P, const DevModel& dm, int t, int D, int pmf_off, const double* Vn,
                      double* Vt, int* Qt, long long lo, long long hi, cudaStream_t stream) {
    if (hi <= lo) return SDPB_OK;
    ColArgs a;
    a.t = t; a.D = D; a.pmf_off = pmf_off; a.Vn = Vn; a.Vt = Vt; a.Qt = Qt; a.lo = lo; a.hi = hi;
    a.A = dm.max_order_idx + 1; a.NQB = P.NQB; a.LT = P.LT; a.di_max = P.di_max; a.NRW = P.NRW;
    a.nthreads = P.nthreads;
    a.nq2_groups = dm.lead == 2 ? (dm.nQ + P.NQB - 1) / P.NQB : 1;
    const int n_levels = DEDUP ? dm.nI + dm.nQ - 1 : dm.nQ;
    a.n_ltiles = (n_levels + P.LT - 1) / P.LT;
    long long rows = 1;
    a.row0 = 0;
    if (!DEDUP) {
        const long long per_x = dm.lead == 2 ? (long long)dm.nQ * dm.nQ : (long long)dm.nQ;
        a.row0 = lo / per_x;
        rows = (hi - 1) / per_x - a.row0 + 1;
    }
    const long long blocks = rows * a.n_ltiles * a.nq2_groups;
    const bool last = (Vn == nullptr), mn = dm.is_min != 0;  // period T without a terminal table
    cudaError_t e = cudaSuccess;
#define SDPB_COL_LAUNCH(MN, LS)                                                                        \
    {                                                                                                  \
        auto k = bi_lead_col<MN, LS, DEDUP>;                                                           \
        if (P.smem > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.smem); \
        if (e == cudaSuccess) k<<<(unsigned)blocks, P.nthreads, P.smem, stream>>>(dm, a);              \
    }
    if (mn) { if (last) SDPB_COL_LAUNCH(true, true) else SDPB_COL_LAUNCH(true, false) }
    else    { if (last) SDPB_COL_LAUNCH(false, true) else SDPB_COL_LAUNCH(false, false) }
#undef SDPB_COL_LAUNCH
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    return SDPB_OK;
}

// ---- action slices over separate CTAs (bi_cash_diag, bi_cash_int, bi_lead_q2m): one merge kernel ----
// Optimum over the action slices of one state: slices in ascending order hold ascending actions, so a strict compare
// keeps the first optimum (Recursion.java:146-157); a slice that held no feasible action of the state says kNoAction.
// A peer shard's V tables as this shard addresses them: V_t[idx] of the peer is at base0 + (t-1)*stride + idx*8 (the
// base is biased by the peer's window start), and the peer reads rows [lo, hi) of this shard's block.
struct DevPeer { char* base0; unsigned long long stride; long long lo, hi; };

// Multi-GPU: the merged values a peer reads are stored into the peer's table as well (peer-mapped memory), so the
// cash models -- where every shard reads nearly every row: 7 peers at 8 GPUs -- need no copy after the kernel either.
template <bool IS_MIN>
__global__ void __launch_bounds__(256)
merge_action_slices(const double* __restrict__ sv, const int* __restrict__ sa, int parts, long long n_local,
                    double* __restrict__ Vt, int* __restrict__ Qt, long long lo, const DevPeer* __restrict__ peers,
                    int n_peers, int t) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_local) return;
    double best = IS_MIN ? DBL_MAX : -DBL_MAX;
    int arg = kNoAction;
    for (int q = 0; q < parts; q++) {
        const double v = sv[(long long)q * n_local + i];
        const int av = sa[(long long)q * n_local + i];
        if (av != kNoAction && (IS_MIN ? (v < best) : (v > best))) { best = v; arg = av; }
    }
    Vt[i] = best;
    Qt[i] = arg == kNoAction ? -1 : arg;
    const long long idx = lo + i;
    for (int p = 0; p < n_peers; p++) {
        const DevPeer pr = peers[p];
        if (idx >= pr.lo && idx < pr.hi)
            reinterpret_cast<double*>(pr.base0 + (unsigned long long)(t - 1) * pr.stride)[idx] = best;
    }
}

// ---------------------------------------------------------------------------------------------
// bi_lead_q2 — lead time 2, every action inside the thread (no cross-thread argopt, no barrier).
//
// A thread owns YT = 8 consecutive preQ1 levels of one (x, preQ2) and walks ALL actions itself, keeping
// the running optimum of its 8 states in registers.  For a fixed action the successor of slot k at
// demand j is (x + l0 + k - d_j, preQ2, a): the same sliding window along the level axis as in
// bi_lead_col.  Lanes hold consecutive preQ2, so the successor table is read TRANSPOSED,
//     VnT[(il * nQ + a) * nQ + preQ2]  =  V_{t+1}[(il * nQ + preQ2) * nQ + a]
// (transpose_q2a, one 16 B/state pass per period), which makes every gather a coalesced row segment
// and every V_t / Q_t store coalesced as well.  Threads are numbered flat over (x, chunk, preQ2) so no
// lane idles on the 101-wide axes; a CTA's threads span at most a few inventory rows and share one
// shared-memory table of (level cost, successor row offset) over the levels they can reach.
// The register window has W = YT + PF entries for both the costs and the successor values, so each
// load lands in its final register PF + 1 demand steps before its first use (as in bi_cash_diag).
// fp64 per evaluation: (1 + 4*8) / 8 = 4.125 (2.125 in the last period), as bi_lead_col, but the
// 8 x NQB shared-memory argopt, its barrier and the one-CTA-per-SM occupancy are gone.  (A warp-per-chunk
// numbering that lets a CTA's warps share successor rows in L1 was measured slower: 149-175 ms vs 140 on C4.  So was a
// variant with TWO actions per pass of the demand loop -- shared LDS.128 and row offsets, 66 fp64 instructions per step
// against ~8 others -- at 168 registers and 3 CTAs per SM: 146.5 vs 141.9 ms.)
struct Q2Args {
    int t, D, pmf_off;
    const double* VnT;        // transposed V_{t+1} (nullptr in the last period)
    double* Vt;
    int* Qt;
    long long lo, hi;
    long long f_begin, f_end; // flat thread range: f = (x * n_chunks + chunk) * nQ + preQ2
    int n_chunks, tpx;        // chunks of 8 levels along preQ1; threads per inventory row
    int cs;                   // bi_lead_q2m: ceil(nQ / 3), the distance between a thread's preQ2 columns
    double* slice_v;          // bi_lead_q2m with the action range cut over gridDim.y: [slice][hi - lo] optima, merged by
    int* slice_a;             // merge_action_slices (which also stores the peers' rows)
    int di_max, NRW;
    int parts;                // slices of the action range per CTA (1, 2 or 4): small grids cannot fill the GPU otherwise
    // Multi-GPU: rows of this shard's block that a peer reads are stored into the peer's V_t as well, straight from the
    // epilogue through peer-mapped memory (the pointers are biased like Vt: indexed by the absolute flattened index),
    // so the hand-over needs no copy after the kernel -- the NVLink writes overlap the arithmetic of the other CTAs.
    int n_peer;
    double* peer_v[2];
    long long peer_lo[2], peer_hi[2];
};

struct PeerStore { double* v; long long lo, hi; };

constexpr int kQ2YT = 8, kQ2PF = 2, kQ2PAD = kQ2PF + 1;

__global__ void transpose_q2a(const double* __restrict__ V, double* __restrict__ VT, int nQ, int row0) {
    __shared__ double tile[32][33];
    const long long base = (long long)(row0 + blockIdx.x) * nQ * nQ;
    const int c0 = blockIdx.y * 32, r0 = blockIdx.z * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int row = r0 + r, c = c0 + threadIdx.x;
        if (row < nQ && c < nQ) tile[r][threadIdx.x] = V[base + (long long)row * nQ + c];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int row = c0 + r, c = r0 + threadIdx.x;  // transposed coordinates
        if (row < nQ && c < nQ) VT[base + (long long)row * nQ + c] = tile[threadIdx.x][r];
    }
}

template <bool IS_MIN, bool LAST, int NT, int PARTS>
__global__ void __launch_bounds__(NT, 512 / NT)
bi_lead_q2(const __grid_constant__ DevModel M, const __grid_constant__ Q2Args a) {
    constexpr int YT = kQ2YT, PF = kQ2PF, W = YT + PF, PAD = kQ2PAD;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* WR = reinterpret_cast<double2*>(smem_raw);  // (level cost, successor row offset in the low word)
    double2* PP = WR + a.NRW;                            // (p, p*gamma)
    const int D = a.D, nQ = M.nQ, tid = threadIdx.x;
    constexpr int cols = NT / PARTS;
    const int part = tid / cols, col = tid - part * cols;
    double* MV = reinterpret_cast<double*>(PP + D);      // [PARTS-1][YT][cols] optima of the action slices > 0
    int* MA = reinterpret_cast<int*>(MV + (size_t)(PARTS - 1) * YT * cols);
    const long long F0 = a.f_begin + (long long)blockIdx.x * cols;
    const long long x_first = F0 / a.tpx;
    const bool lost = (M.flags & SDPB_F_LOST_SALES) != 0;

    for (int j = tid; j < D; j += NT) PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
    // window index wi <-> unclamped level index il = x_first - di_max - PAD + wi
    for (int wi = tid; wi < a.NRW; wi += NT) {
        const long long il = x_first - a.di_max - PAD + wi;
        const double lvl = M.inv_min + (double)il * M.step;
        long long is = il;
        if (lost) is = is > M.i_zero ? is : M.i_zero;
        is = is < M.nI - 1 ? is : M.nI - 1;  // upper clamp first; also the memory-safety clip
        is = is > 0 ? is : 0;
        WR[wi] = make_double2(M.h * fmax(lvl, 0.0) + M.pen * fmax(-lvl, 0.0),
                              __hiloint2double(0, (int)(is * nQ * nQ)));
    }
    __syncthreads();

    const long long F = min(F0 + col, a.f_end - 1);
    const long long x = F / a.tpx;
    const int f = (int)(F - x * a.tpx);
    const int chunk = f / nQ, q2 = f - chunk * nQ, l0 = chunk * YT;
    const long long idx0 = (x * nQ + l0) * nQ + q2;  // slot k: idx0 + k * nQ
    bool any = false;
#pragma unroll
    for (int k = 0; k < YT; k++) any |= (l0 + k < nQ) && idx0 + (long long)k * nQ >= a.lo && idx0 + (long long)k * nQ < a.hi;
    any = any && F0 + col < a.f_end;
    if (PARTS == 1 && !any) return;

    // slot k at demand j reads window row  (x - x_first) + l0 + k + (D-1-j) + PAD
    const unsigned wr0 = (unsigned)__cvta_generic_to_shared(WR) + (unsigned)((int)(x - x_first) + l0 + (D - 1) + PAD) * 16u;
    const unsigned pp_s = (unsigned)__cvta_generic_to_shared(PP);
    const double* __restrict__ cb = LAST ? nullptr : a.VnT + q2;
    const double vt = M.v_t[a.t - 1];

    double best[YT];
    int arg[YT];
#pragma unroll
    for (int k = 0; k < YT; k++) { best[k] = IS_MIN ? DBL_MAX : -DBL_MAX; arg[k] = kNoAction; }

    const int per_part = (M.max_order_idx + PARTS) / PARTS;  // ceil(A / PARTS)
    const int ai_begin = any ? part * per_part : 0;
    const int ai_end = any ? min(M.max_order_idx + 1, ai_begin + per_part) : 0;
    if (!LAST) cb += (long long)ai_begin * nQ;
    for (int ai = ai_begin; ai < ai_end; ai++) {
        const double av = (double)ai * M.step;
        const double fv = (av > 0.0 ? M.K : 0.0) + vt * av;  // Leadtime.java:73-74,79
        double acc[YT], cst[W], Vw[W];
#pragma unroll
        for (int k = 0; k < YT; k++) acc[k] = 0.0;
#pragma unroll
        for (int k = 0; k < W; k++) {  // entries YT..W-1: the levels slot 0 reaches at demands PF..1
            const double2 e = lds_double2(wr0 + (unsigned)((k < YT ? k : k - W) * 16));
            cst[k] = fv + e.x;
            Vw[k] = LAST ? 0.0 : __ldg(cb + __double2loint(e.y));
        }
        unsigned wr_run = wr0 - (unsigned)((PF + 1) * 16);
#define SDPB_Q2_STEP(JJ)                                                                              \
        {                                                                                                 \
            const double2 pp = lds_double2(pp_s + (unsigned)j * 16u);                                     \
            _Pragma("unroll") for (int k = 0; k < YT; k++) {                                              \
                acc[k] += pp.x * cst[(k - (JJ) + W) % W];          /* LeadtimeRecursion.java:59 */       \
                if (!LAST) acc[k] += pp.y * Vw[(k - (JJ) + W) % W]; /* LeadtimeRecursion.java:62 */      \
            }                                                                                             \
            const double2 e = lds_double2(wr_run);   /* refill the entry slot 7 just released */          \
            cst[(YT - 1 - (JJ) + W) % W] = fv + e.x;                                                      \
            if (!LAST) Vw[(YT - 1 - (JJ) + W) % W] = __ldg(cb + __double2loint(e.y));                     \
            wr_run -= 16u;                                                                                \
            j += 1;                                                                                       \
        }
        int j = 0;
        while (j + W <= D) {
#pragma unroll
            for (int JJ = 0; JJ < W; JJ++) SDPB_Q2_STEP(JJ)
        }
#pragma unroll
        for (int JJ = 0; JJ < W - 1; JJ++)
            if (j < D) SDPB_Q2_STEP(JJ)
#undef SDPB_Q2_STEP
#pragma unroll
        for (int k = 0; k < YT; k++)
            if (IS_MIN ? (acc[k] < best[k]) : (acc[k] > best[k])) { best[k] = acc[k]; arg[k] = ai; }
        if (!LAST) cb += nQ;
    }
    if (PARTS > 1) {
        if (part > 0) {
#pragma unroll
            for (int k = 0; k < YT; k++) {
                MV[((part - 1) * YT + k) * cols + col] = best[k];
                MA[((part - 1) * YT + k) * cols + col] = arg[k];
            }
        }
        __syncthreads();
        if (part > 0 || !any) return;
        for (int q = 0; q < PARTS - 1; q++) {  // ascending slices hold ascending actions: strict compare = first wins
#pragma unroll
            for (int k = 0; k < YT; k++) {
                const double v = MV[(q * YT + k) * cols + col];
                const int av = MA[(q * YT + k) * cols + col];
                if (av != kNoAction && (IS_MIN ? (v < best[k]) : (v > best[k]))) { best[k] = v; arg[k] = av; }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < YT; k++) {
        const long long idx = idx0 + (long long)k * nQ;
        if (l0 + k < nQ && idx >= a.lo && idx < a.hi) {
            a.Vt[idx] = best[k];
            a.Qt[idx] = arg[k] == kNoAction ? -1 : arg[k];
            for (int p = 0; p < a.n_peer; p++)
                if (idx >= a.peer_lo[p] && idx < a.peer_hi[p]) a.peer_v[p][idx] = best[k];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// bi_lead_q2m -- bi_lead_q2 with the products p_j * (fv_a + L(level)) shared by the threads of a CTA, and the demand loop
// walked along level diagonals.
//
// The immediate value of (x, preQ1, preQ2) under action a and demand d_j does not depend on preQ2
// (Leadtime.java:72-80: fixed + variable + holding/penalty of x + preQ1 - d_j), and the lanes of a warp ARE consecutive
// preQ2 of one (x, chunk of 8 preQ1 levels): all of them form the identical product m = p_j * cst for each of their 8
// slots.  A CTA tabulates these products once per action for the few (x, chunk) groups its threads belong to (5 on C4)
// with exactly the operations a thread used to do itself, and a thread reads them back and spends (add, mul, add) per
// evaluation instead of (mul, add, mul, add) + 1/8.
//
// Demands are consecutive (d_j = d_0 + j), so slot k at demand j reads the successor level x + l0 + k - d_0 - j.  The
// demand loop runs over diagonals n = j - k + 7 (n = 0 .. D + 6) instead of over j: on diagonal n every slot k that has
// a demand j = n - 7 + k in [0, D) reads the SAME level u_n = x + l0 - d_0 - n + 7.  So per diagonal a thread gathers one
// successor value per column, and reads the 8 products M[group][n][k] = p_{n-7+k} * (fv_a + L(u_n)) with four LDS.128;
// p*gamma for slot k is p_{n-7+k}*gamma, a sliding window that all columns share.  The first 7 and the last 7 diagonals
// have fewer active slots, known at compile time; demand supports shorter than 7 take a plain loop that tests each slot.
// Each state still adds its terms for j = 0, 1, ..., D-1 in order with the same operands: values are bit-identical.
//
// Registers: 8*NC accumulators, an 8-entry p*gamma window and 2*NC prefetched successor values, so a thread owns THREE
// preQ2 columns (c, c + cs, c + 2*cs with cs = ceil(nQ/3): lanes stay consecutive, every gather a coalesced row segment)
// -- 24 states, 72 fp64 instructions per diagonal against 4 + 1 LDS.128 and 3 gathers.  The running optimum of the 24
// states lives in shared memory (read-compare-conditional-store once per action; the action as 16 bits, since plan_q2
// keeps nQ below 46341).  The per-diagonal refill (p*gamma entering the window, successor row offset two diagonals
// ahead) comes from a second table R[group][n], built once per CTA.  M is single-buffered -- two barriers per action --
// which keeps the tables of C4 at 45 KB, four CTAs per SM.
template <int IMM>
__device__ __forceinline__ double2 lds_double2_o(unsigned shared_addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2+%3];" : "=d"(v.x), "=d"(v.y) : "r"(shared_addr), "n"(IMM));
    return v;
}

constexpr int kQ2mNC = 3;   // preQ2 columns per thread
constexpr int kQ2mPW = kQ2YT;  // p*gamma window: one entry per slot
constexpr unsigned short kQ2mNoAction = 0xffff;

struct Q2mLayout { int NG; unsigned off_rg, off_gb, off_pz, off_bv, off_ba, off_mt; size_t smem; };

__host__ __device__ inline Q2mLayout q2m_layout(int NRW, int D, int NT, int cs) {
    Q2mLayout L;
    L.NG = (NT - 1) / cs + 2;                                    // distinct (x, chunk) groups among NT consecutive threads
    const unsigned R = (unsigned)(D + kQ2YT - 1);                // diagonals per group
    unsigned o = (unsigned)(NRW + D) * 16u;                      // WR, PP
    L.off_rg = o; o += (unsigned)L.NG * R * 16u;                 // R[group][n] = (p_{n+1}*gamma, row offset of u_{n+2})
    L.off_gb = o; o += ((unsigned)L.NG * 4u + 15u) & ~15u;       // window row of each group's level u_7
    L.off_pz = o; o += ((R + kQ2YT - 1) * 8u + 15u) & ~15u;      // p_j for j = -7 .. D+6, zero outside [0, D)
    L.off_bv = o; o += (unsigned)(kQ2mNC * kQ2YT * NT) * 8u;     // running optimum per state: value ...
    L.off_ba = o; o += ((unsigned)(kQ2mNC * kQ2YT * NT) * 2u + 15u) & ~15u;  // ... and action
    L.off_mt = o; o += (unsigned)L.NG * R * 64u;                 // M[group][n][8]
    L.smem = o;
    return L;
}

// Diagonal n of one action: slots [KLO, KHI) add their term, p*gamma of slot k in pw[(PH + k) % kQ2mPW], the successor
// value of column c in vb[c][VS], the products at mt + IMM.
template <bool LAST, int KLO, int KHI, int PH, int VS, int IMM>
__device__ __forceinline__ void q2m_diag(double (&acc)[kQ2mNC][kQ2YT], unsigned mt, const double (&pw)[kQ2mPW],
                                         const double (&vb)[kQ2mNC][2]) {
    double mm[kQ2YT];
    if (KLO < 2 && KHI > 0) { const double2 t = lds_double2_o<IMM>(mt); mm[0] = t.x; mm[1] = t.y; }
    if (KLO < 4 && KHI > 2) { const double2 t = lds_double2_o<IMM + 16>(mt); mm[2] = t.x; mm[3] = t.y; }
    if (KLO < 6 && KHI > 4) { const double2 t = lds_double2_o<IMM + 32>(mt); mm[4] = t.x; mm[5] = t.y; }
    if (KLO < 8 && KHI > 6) { const double2 t = lds_double2_o<IMM + 48>(mt); mm[6] = t.x; mm[7] = t.y; }
#pragma unroll
    for (int k = KLO; k < KHI; k++)
#pragma unroll
        for (int c = 0; c < kQ2mNC; c++) {
            acc[c][k] += mm[k];                                            // LeadtimeRecursion.java:59
            if (!LAST) acc[c][k] += pw[(PH + k) % kQ2mPW] * vb[c][VS];    // LeadtimeRecursion.java:62
        }
}

// After diagonal n: R[group][n] at rg + IMM gives p_{n+1}*gamma (into pw[PS]; PS < 0 drops it) and the successor row
// of diagonal n + 2, whose values go to vb[.][VS].
template <int VS, int PS, int IMM>
__device__ __forceinline__ void q2m_refill(double (&pw)[kQ2mPW], double (&vb)[kQ2mNC][2], unsigned rg,
                                           const double* const (&cb)[kQ2mNC]) {
    const double2 r = lds_double2_o<IMM>(rg);
    if (PS >= 0) pw[PS < 0 ? 0 : PS] = r.x;
    const unsigned off = (unsigned)__double2loint(r.y);
#pragma unroll
    for (int c = 0; c < kQ2mNC; c++) vb[c][VS] = __ldg(cb[c] + off);
}

template <bool IS_MIN, bool LAST, int NT>
__global__ void __launch_bounds__(NT, 512 / NT)
bi_lead_q2m(const __grid_constant__ DevModel M, const __grid_constant__ Q2Args a) {
    constexpr int YT = kQ2YT, PAD = kQ2PAD, NC = kQ2mNC, PW = kQ2mPW;
    static_assert(YT == 8 && NC == 3 && PW == 8, "the diagonals below are written out for these sizes");
    static_assert(NT % 8 == 0, "the table builder keeps the slot index fixed per thread");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int D = a.D, nQ = M.nQ, cs = a.cs, tid = threadIdx.x;
    const int R = D + YT - 1;                            // diagonals
    const Q2mLayout L = q2m_layout(a.NRW, D, NT, cs);
    double2* WR = reinterpret_cast<double2*>(smem_raw);  // (level cost, successor row offset in the low word)
    double2* PP = WR + a.NRW;                            // (p, p*gamma)
    double2* RG = reinterpret_cast<double2*>(smem_raw + L.off_rg);
    int* GB = reinterpret_cast<int*>(smem_raw + L.off_gb);
    double* PZ = reinterpret_cast<double*>(smem_raw + L.off_pz);  // PZ[n + k] = p_{n-7+k}: slot k on diagonal n
    double* BV = reinterpret_cast<double*>(smem_raw + L.off_bv);
    unsigned short* BA = reinterpret_cast<unsigned short*>(smem_raw + L.off_ba);
    double* MT = reinterpret_cast<double*>(smem_raw + L.off_mt);
    const int NG = L.NG;
    const long long F0 = a.f_begin + (long long)blockIdx.x * NT;
    const long long x_first = F0 / a.tpx;
    const long long G0 = F0 / cs;                        // first (x, chunk) group of the CTA: G = x * n_chunks + chunk
    const bool lost = (M.flags & SDPB_F_LOST_SALES) != 0;

    for (int j = tid; j < D; j += NT) PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
    for (int j = tid; j < R + YT - 1; j += NT) {
        const int jd = j - (YT - 1);
        PZ[j] = jd >= 0 && jd < D ? M.pmf_p[a.pmf_off + jd] : 0.0;
    }
    for (int wi = tid; wi < a.NRW; wi += NT) {
        const long long il = x_first - a.di_max - PAD + wi;
        const double lvl = M.inv_min + (double)il * M.step;
        long long is = il;
        if (lost) is = is > M.i_zero ? is : M.i_zero;
        is = is < M.nI - 1 ? is : M.nI - 1;  // upper clamp first; also the memory-safety clip
        is = is > 0 ? is : 0;
        WR[wi] = make_double2(M.h * fmax(lvl, 0.0) + M.pen * fmax(-lvl, 0.0),
                              __hiloint2double(0, (int)(is * nQ * nQ)));
    }
    // window row of u_7 (slot 0 at demand D-1) for each group; diagonal n reads row GB + 7 - n
    for (int g = tid; g < NG; g += NT) {
        const long long G = G0 + g;
        const long long xg = G / a.n_chunks;
        const int chunk = (int)(G - xg * a.n_chunks);
        int wb = (int)(xg - x_first) + chunk * YT + (D - 1) + PAD;
        GB[g] = min(wb, a.NRW - YT);  // groups past the end of the range are built but never read
    }
#pragma unroll
    for (int s2 = 0; s2 < NC * YT; s2++) { BV[s2 * NT + tid] = IS_MIN ? DBL_MAX : -DBL_MAX; BA[s2 * NT + tid] = kQ2mNoAction; }
    __syncthreads();
    for (int e = tid; e < NG * R; e += NT) {
        const int g = e / R, n = e - g * R;
        RG[e] = make_double2(n + 1 < D ? PP[n + 1].y : 0.0, WR[GB[g] + 5 - n].y);
    }

    const long long F = min(F0 + tid, a.f_end - 1);
    const long long x = F / a.tpx;
    const int f = (int)(F - x * a.tpx);
    const int chunk = f / cs, c0 = f - chunk * cs, l0 = chunk * YT;
    const int g_own = (int)(F / cs - G0);
    const long long idx0 = (x * nQ + l0) * nQ + c0;      // column c, slot k: idx0 + k * nQ + c * cs
    // the thread's states span [idx0, idx_end]; one in [lo, hi) makes it compute (the stores below test each state)
    const long long idx_end = idx0 + (long long)(min(YT, nQ - l0) - 1) * nQ + (long long)((nQ - 1 - c0) / cs) * cs;
    const bool any = F0 + tid < a.f_end && idx_end >= a.lo && idx0 < a.hi;

    const unsigned wr_s = (unsigned)__cvta_generic_to_shared(WR);
    const unsigned pp_s = (unsigned)__cvta_generic_to_shared(PP);
    const unsigned rg0 = (unsigned)__cvta_generic_to_shared(RG) + (unsigned)(g_own * R) * 16u;
    const unsigned mt0 = (unsigned)__cvta_generic_to_shared(MT) + (unsigned)(g_own * R) * 64u;
    const unsigned bv_s = (unsigned)__cvta_generic_to_shared(BV) + (unsigned)tid * 8u;
    const unsigned ba_s = (unsigned)__cvta_generic_to_shared(BA) + (unsigned)tid * 2u;
    const int gb = (int)(x - x_first) + l0 + (D - 1) + PAD;  // this thread's window row of u_7
    const double* cb[NC];  // the successor row of each column under action ai; a missing column gathers the first one
#pragma unroll
    for (int c = 0; c < NC; c++) cb[c] = LAST ? nullptr : a.VnT + c0 + (c0 + c * cs < nQ ? c * cs : 0);
    const double vt = M.v_t[a.t - 1];

    // the action range, cut over gridDim.y (separate CTAs, merged by merge_action_slices: small grids need more CTAs
    // than their states give)
    const int n_sl = (int)gridDim.y, sl = (int)blockIdx.y;
    const int per_sl = (M.max_order_idx + n_sl) / n_sl;      // ceil(A / n_sl)
    const int ai_begin = sl * per_sl, ai_end = min(M.max_order_idx + 1, ai_begin + per_sl);
#pragma unroll
    for (int c = 0; c < NC; c++) if (!LAST) cb[c] += (long long)ai_begin * nQ;
    for (int ai = ai_begin; ai < ai_end; ai++) {
        {  // ---- tabulate p_j * (fv_a + L(u_n)) for the CTA's groups, j = n - 7 + k: a thread per (group, diagonal) ----
            const double av = (double)ai * M.step;
            const double fv = (av > 0.0 ? M.K : 0.0) + vt * av;  // Leadtime.java:73-74,79
            for (int r = tid; r < NG * R; r += NT) {
                const int g = r / R, n = r - g * R;
                const double cst = fv + WR[GB[g] + (YT - 1) - n].x;
                double2* Mr = reinterpret_cast<double2*>(MT + (size_t)r * YT);
#pragma unroll
                for (int k = 0; k < YT; k += 2)                   // LeadtimeRecursion.java:59
                    Mr[k / 2] = make_double2(PZ[n + k] * cst, PZ[n + k + 1] * cst);
            }
        }
        __syncthreads();
        if (any) {
            double acc[NC][YT];
#pragma unroll
            for (int c = 0; c < NC; c++)
#pragma unroll
                for (int k = 0; k < YT; k++) acc[c][k] = 0.0;
            if (D >= YT - 1) {
                double pw[PW], vb[NC][2];
                if (!LAST) {  // p_0 * gamma, and the successor values of diagonals 0 and 1
                    pw[0] = lds_double(pp_s + 8u);
#pragma unroll
                    for (int n = 0; n < 2; n++) {
                        const unsigned off = (unsigned)__double2loint(lds_double(wr_s + (unsigned)(gb + 7 - n) * 16u + 8u));
#pragma unroll
                        for (int c = 0; c < NC; c++) vb[c][n] = __ldg(cb[c] + off);
                    }
                }
#define SDPB_Q2M_HEAD(N)                                                                              \
                q2m_diag<LAST, YT - 1 - (N), YT, (N) + 1, (N) & 1, (N) * 64>(acc, mt0, pw, vb);           \
                if (!LAST) q2m_refill<(N) & 1, (N) + 1, (N) * 16>(pw, vb, rg0, cb);
                SDPB_Q2M_HEAD(0) SDPB_Q2M_HEAD(1) SDPB_Q2M_HEAD(2) SDPB_Q2M_HEAD(3)
                SDPB_Q2M_HEAD(4) SDPB_Q2M_HEAD(5) SDPB_Q2M_HEAD(6)
#undef SDPB_Q2M_HEAD
                // all slots active: diagonals 7 .. D-1, in blocks of PW that start at an odd n, so the window position
                // of step U of a block is U and its successor values sit in vb[.][(U + 1) & 1]
#define SDPB_Q2M_FULL(U)                                                                              \
                q2m_diag<LAST, 0, YT, (U), ((U) + 1) & 1, (U) * 64>(acc, mt_run, pw, vb);                 \
                if (!LAST) q2m_refill<((U) + 1) & 1, (U), (U) * 16>(pw, vb, rg_run, cb);
                int n = YT - 1;
                unsigned mt_run = mt0 + (unsigned)n * 64u, rg_run = rg0 + (unsigned)n * 16u;
                for (; n + PW <= D; n += PW, mt_run += PW * 64u, rg_run += PW * 16u) {
                    SDPB_Q2M_FULL(0) SDPB_Q2M_FULL(1) SDPB_Q2M_FULL(2) SDPB_Q2M_FULL(3) SDPB_Q2M_FULL(4)
                    SDPB_Q2M_FULL(5) SDPB_Q2M_FULL(6) SDPB_Q2M_FULL(7)
                }
                if (n + 0 < D) { SDPB_Q2M_FULL(0) }
                if (n + 1 < D) { SDPB_Q2M_FULL(1) }
                if (n + 2 < D) { SDPB_Q2M_FULL(2) }
                if (n + 3 < D) { SDPB_Q2M_FULL(3) }
                if (n + 4 < D) { SDPB_Q2M_FULL(4) }
                if (n + 5 < D) { SDPB_Q2M_FULL(5) }
                if (n + 6 < D) { SDPB_Q2M_FULL(6) }
                if (n + 7 < D) { SDPB_Q2M_FULL(7) }
#undef SDPB_Q2M_FULL
                // diagonals D .. D+6, slots k < 7 - e on diagonal D + e.  Where the window stands now depends on D, so
                // p_{D-7..D-1} * gamma are read again, and the values of diagonals D and D+1 picked by the parity of D.
                double pe[PW], ve[NC][2];
                if (!LAST) {
#pragma unroll
                    for (int m = 0; m < YT - 1; m++) pe[m] = lds_double(pp_s + (unsigned)(D - (YT - 1) + m) * 16u + 8u);
                    const bool odd = (D & 1) != 0;
#pragma unroll
                    for (int c = 0; c < NC; c++) {
                        ve[c][0] = odd ? vb[c][1] : vb[c][0];
                        ve[c][1] = odd ? vb[c][0] : vb[c][1];
                    }
                }
                const unsigned mt_d = mt0 + (unsigned)D * 64u, rg_d = rg0 + (unsigned)D * 16u;
#define SDPB_Q2M_TAIL(E)                                                                              \
                q2m_diag<LAST, 0, YT - 1 - (E), (E), (E) & 1, (E) * 64>(acc, mt_d, pe, ve);               \
                if (!LAST && (E) + 2 < YT - 1) q2m_refill<(E) & 1, -1, (E) * 16>(pe, ve, rg_d, cb);
                SDPB_Q2M_TAIL(0) SDPB_Q2M_TAIL(1) SDPB_Q2M_TAIL(2) SDPB_Q2M_TAIL(3)
                SDPB_Q2M_TAIL(4) SDPB_Q2M_TAIL(5) SDPB_Q2M_TAIL(6)
#undef SDPB_Q2M_TAIL
            } else {  // D < 7: every diagonal has both ends cut; test each slot
                for (int n = 0; n < R; n++) {
                    double mm[YT], v[NC];
                    if (!LAST) {
                        const unsigned off = (unsigned)__double2loint(lds_double(wr_s + (unsigned)(gb + 7 - n) * 16u + 8u));
#pragma unroll
                        for (int c = 0; c < NC; c++) v[c] = __ldg(cb[c] + off);
                    }
#pragma unroll
                    for (int p = 0; p < YT / 2; p++) {
                        const double2 t = lds_double2(mt0 + (unsigned)n * 64u + (unsigned)p * 16u);
                        mm[2 * p] = t.x; mm[2 * p + 1] = t.y;
                    }
#pragma unroll
                    for (int k = 0; k < YT; k++) {
                        const int j = n - (YT - 1) + k;
                        if (j < 0 || j >= D) continue;
                        const double pg = LAST ? 0.0 : lds_double(pp_s + (unsigned)j * 16u + 8u);
#pragma unroll
                        for (int c = 0; c < NC; c++) {
                            acc[c][k] += mm[k];                             // LeadtimeRecursion.java:59
                            if (!LAST) acc[c][k] += pg * v[c];              // LeadtimeRecursion.java:62
                        }
                    }
                }
            }
            // running optimum: strictly better wins, so the first (lowest) optimal action stays (Recursion.java:146-157)
#pragma unroll
            for (int c = 0; c < NC; c++)
#pragma unroll
                for (int k = 0; k < YT; k++) {
                    const unsigned so = (unsigned)((c * YT + k) * NT);
                    const double bv = lds_double(bv_s + so * 8u);
                    if (IS_MIN ? (acc[c][k] < bv) : (acc[c][k] > bv)) {
                        asm volatile("st.shared.f64 [%0], %1;" ::"r"(bv_s + so * 8u), "d"(acc[c][k]) : "memory");
                        asm volatile("st.shared.u16 [%0], %1;" ::"r"(ba_s + so * 2u), "h"((unsigned short)ai) : "memory");
                    }
                }
        }
        __syncthreads();  // M is rebuilt for the next action
#pragma unroll
        for (int c = 0; c < NC; c++) if (!LAST) cb[c] += nQ;
    }
    if (!any) return;
    // the thread's states again, from a fresh read of its index: kept from above, they would stay live through the
    // action loop and push its registers into local memory
    unsigned ts;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(ts));
    const long long Fs = min(F0 + (long long)ts, a.f_end - 1);
    const long long xs = Fs / a.tpx;
    const int fs = (int)(Fs - xs * a.tpx);
    const int cks = fs / cs, c0s = fs - cks * cs, l0s = cks * YT;
    const long long idx0s = (xs * nQ + l0s) * nQ + c0s;
#pragma unroll
    for (int c = 0; c < NC; c++) {
        if (c0s + c * cs >= nQ) break;
#pragma unroll
        for (int k = 0; k < YT; k++) {
            const long long idx = idx0s + (long long)k * nQ + c * cs;
            if (!(l0s + k < nQ && idx >= a.lo && idx < a.hi)) continue;
            const double best = BV[(c * YT + k) * NT + ts];
            const unsigned short ba = BA[(c * YT + k) * NT + ts];
            const int arg = ba == kQ2mNoAction ? kNoAction : (int)ba;
            if (n_sl > 1) {  // this CTA saw one slice of the actions only
                a.slice_v[(long long)sl * (a.hi - a.lo) + (idx - a.lo)] = best;
                a.slice_a[(long long)sl * (a.hi - a.lo) + (idx - a.lo)] = arg;
                continue;
            }
            a.Vt[idx] = best;
            a.Qt[idx] = arg == kNoAction ? -1 : arg;
            for (int p = 0; p < a.n_peer; p++)
                if (idx >= a.peer_lo[p] && idx < a.peer_hi[p]) a.peer_v[p][idx] = best;
        }
    }
}

struct Q2Plan {
    bool ok = false;
    int NT = 128, n_chunks = 0, tpx = 0, di_max = 0, NRW = 0;
    size_t smem = 0;
};

inline Q2Plan plan_q2(const sdpb_model& m, const DevModel& d, int D, const int* di) {
    Q2Plan P;
    if (m.cost_kind != SDPB_COST_BACKORDER || m.lead_time != 2) return P;
    for (int j = 0; j < D; j++)
        if (di[j] != di[0] + j) return P;  // the register window needs consecutive demands
    if ((long long)d.nI * d.nQ * d.nQ >= 0x7fffffffLL) return P;  // 32-bit successor row offsets
    P.n_chunks = (d.nQ + kQ2YT - 1) / kQ2YT;
    P.tpx = P.n_chunks * d.nQ;
    P.di_max = di[D - 1];
    const int dx_max = (P.NT + P.tpx - 1) / P.tpx + 1;  // inventory rows a CTA's threads can span
    P.NRW = P.n_chunks * kQ2YT + D + kQ2PAD + dx_max;
    P.smem = (size_t)(P.NRW + D) * 16 + (size_t)kQ2YT * P.NT * 12;  // + the action-slice merge: (parts-1)/parts * YT * NT entries
    P.ok = P.smem <= 96 * 1024;
    return P;
}

// VnT: scratch of nI*nQ*nQ doubles; filled here from Vn (stream order) unless this is the last period.
// [row0, row1): inventory rows of V_{t+1} the range [lo, hi) can read (sdpb_shard_reads); only those are transposed.
constexpr int kQ2MaxPeers = 2;

// How a launch over [lo, hi) is shaped.  bi_lead_q2m (shared products) whenever its tables leave four CTAs per SM (at
// most 56 KB each: an SM has 228 KB of shared memory and keeps 1 KB of it per CTA), with
// the action range cut over separate CTAs (gridDim.y slices, merged by merge_action_slices -- the per-action product
// table is then still built by a full CTA) when the grid is short of ~8 waves; else bi_lead_q2, with the action range cut
// over 2 or 4 thread groups inside a CTA when the grid is short of ~6 waves.
struct Q2Shape { bool shared; int parts, slices, cs, tpx, NRW; long long f_begin, f_end; Q2mLayout L; };

inline Q2Shape q2_shape(const Q2Plan& P, const DevModel& dm, int D, long long lo, long long hi, int sm_count) {
    Q2Shape S{};
    const long long per_x = (long long)dm.nQ * dm.nQ;
    const long long rows = (hi - 1) / per_x - lo / per_x + 1;
    const double waves = (double)(rows * P.tpx) / 32.0 / (16.0 * sm_count);
    S.parts = waves >= 6.0 ? 1 : (waves >= 3.0 ? 2 : 4);
    S.cs = (dm.nQ + kQ2mNC - 1) / kQ2mNC;
    const int tpx2 = P.n_chunks * S.cs;
    const int NRW2 = P.n_chunks * kQ2YT + D + kQ2PAD + (P.NT + tpx2 - 1) / tpx2 + 1;
    S.slices = 1;
    // bi_lead_q2m's threads are numbered over (x, chunk, column triple).  Measured on C4 with two columns
    // per thread (ms, bi_lead_q2m vs bi_lead_q2): whole grid 131.0 vs 140.3.  Shards: with the action range cut over thread groups INSIDE a CTA the per-action tables
    // and the barrier cost more than they save (a quarter of the grid 37.8 vs 36.7, an eighth 20.8 vs 18.7); cut over
    // SEPARATE CTAs they do not (34.1 and 17.7; 2 / 4 / 8 / 16 slices on the eighth: 18.4 / 17.5 / 17.7 / 18.0), so that
    // is the shape every launch takes when the tables fit.  With three columns (B200, 1000 W): whole grid 117.5 ms with
    // the 2 slices this rule gives it (an earlier build of the kernel: 121.0 sliced, 123.1 unsliced); slowest shard of
    // 2 / 4 / 8: 61.2 / 31.6 / 16.6 ms.
    S.L = q2m_layout(NRW2, D, P.NT, S.cs);
    // Test hooks, read once per process: they force shapes that small instances do not take by themselves.
    //   SDPB_Q2_SHARE=1      bi_lead_q2m with no action slices wherever its tables fit: the epilogue with peer stores
    //                        that large shards take
    //   SDPB_Q2_SPLIT=2 | 4  bi_lead_q2 with 2 or 4 thread groups, no shared products
    static const bool force_share = std::getenv("SDPB_Q2_SHARE") != nullptr;
    static const int force_split = [] { const char* e = std::getenv("SDPB_Q2_SPLIT"); return e ? std::atoi(e) : 0; }();
    if (force_split) {
        S.parts = force_split == 2 ? 2 : 4;
    } else if (S.L.smem <= 56 * 1024) {
        S.shared = true; S.parts = 1;
        const double ctas = (double)(rows * tpx2) / P.NT;
        const double w = ctas / (4.0 * sm_count);                // CTA waves at four CTAs per SM
        if (w < 8.0 && !force_share) S.slices = (int)std::min(8.0, std::ceil(8.0 / std::max(w, 0.01)));
        S.slices = std::max(1, std::min(S.slices, (dm.max_order_idx + 1) / 8));
        const int per = (dm.max_order_idx + S.slices) / S.slices;  // as the kernel cuts: no empty slice
        S.slices = (dm.max_order_idx + per) / per;
    }
    S.tpx = S.shared ? tpx2 : P.tpx;
    S.NRW = S.shared ? NRW2 : P.NRW;
    S.f_begin = (lo / per_x) * S.tpx;
    S.f_end = ((hi - 1) / per_x + 1) * S.tpx;
    return S;
}

// S = q2_shape(P, ..., lo, hi, ...).  SDPB_OK, SDPB_ERR_NOMEM (slice scratch too small) or SDPB_ERR_CUDA.
inline int launch_q2(const Q2Plan& P, const Q2Shape& S, const DevModel& dm, int t, int D, int pmf_off, const double* Vn,
                     double* VnT, double* Vt, int* Qt, long long lo, long long hi, int row0, int row1, cudaStream_t stream,
                     const PeerStore* peers, int n_peers, double* slice_v, int* slice_a, size_t slice_cap,
                     const DevPeer* d_peers, int n_dev_peers) {
    if (hi <= lo) return SDPB_OK;
    const bool last = (Vn == nullptr), mn = dm.is_min != 0;  // period T without a terminal table
    if (!last) {
        const unsigned tiles = (unsigned)((dm.nQ + 31) / 32);
        transpose_q2a<<<dim3((unsigned)(row1 - row0), tiles, tiles), dim3(32, 8), 0, stream>>>(Vn, VnT, dm.nQ, row0);
    }
    const long long n_local = hi - lo;
    if (S.slices > 1 && (size_t)S.slices * (size_t)n_local > slice_cap) return SDPB_ERR_NOMEM;  // the caller sizes it: q2_shape
    Q2Args a;
    a.t = t; a.D = D; a.pmf_off = pmf_off; a.VnT = last ? nullptr : VnT; a.Vt = Vt; a.Qt = Qt; a.lo = lo; a.hi = hi;
    a.n_chunks = P.n_chunks; a.tpx = S.tpx; a.di_max = P.di_max; a.NRW = S.NRW;
    a.f_begin = S.f_begin; a.f_end = S.f_end; a.parts = S.parts; a.cs = S.cs;
    a.slice_v = slice_v; a.slice_a = slice_a;
    a.n_peer = 0;
    for (int p = 0; p < kQ2MaxPeers; p++) { a.peer_v[p] = nullptr; a.peer_lo[p] = a.peer_hi[p] = 0; }
    if (S.slices == 1)  // (a sliced launch leaves the peers' rows to the merge kernel)
        for (int p = 0; p < n_peers && p < kQ2MaxPeers; p++) {
            a.peer_v[p] = peers[p].v; a.peer_lo[p] = peers[p].lo; a.peer_hi[p] = peers[p].hi;
            a.n_peer = p + 1;
        }
    const int cols = P.NT / a.parts;
    const Q2mLayout L = S.L;
    const bool shared = S.shared;
    cudaError_t e = cudaSuccess;
    const dim3 grid((unsigned)((a.f_end - a.f_begin + cols - 1) / cols), (unsigned)S.slices);
#define SDPB_Q2_LAUNCH(K, SMEM, GRID)                                                                  \
    {                                                                                                  \
        auto k = K;                                                                                    \
        if (SMEM > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM); \
        if (e == cudaSuccess) k<<<GRID, 128, SMEM, stream>>>(dm, a);                                   \
    }
#define SDPB_Q2_NT(MN, LS)                                                                             \
    if (shared) SDPB_Q2_LAUNCH((bi_lead_q2m<MN, LS, 128>), L.smem, grid)                               \
    else if (a.parts == 1) SDPB_Q2_LAUNCH((bi_lead_q2<MN, LS, 128, 1>), P.smem, grid.x)                \
    else if (a.parts == 2) SDPB_Q2_LAUNCH((bi_lead_q2<MN, LS, 128, 2>), P.smem, grid.x)                \
    else SDPB_Q2_LAUNCH((bi_lead_q2<MN, LS, 128, 4>), P.smem, grid.x)
    if (mn) { if (last) SDPB_Q2_NT(true, true) else SDPB_Q2_NT(true, false) }
    else    { if (last) SDPB_Q2_NT(false, true) else SDPB_Q2_NT(false, false) }
#undef SDPB_Q2_NT
#undef SDPB_Q2_LAUNCH
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    if (S.slices > 1) {
        const unsigned mb = (unsigned)((n_local + 255) / 256);
        if (mn) merge_action_slices<true><<<mb, 256, 0, stream>>>(slice_v, slice_a, S.slices, n_local, Vt + lo, Qt + lo, lo, d_peers, n_dev_peers, t);
        else merge_action_slices<false><<<mb, 256, 0, stream>>>(slice_v, slice_a, S.slices, n_local, Vt + lo, Qt + lo, lo, d_peers, n_dev_peers, t);
        if (cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    }
    return SDPB_OK;
}

}  // namespace sdpb
