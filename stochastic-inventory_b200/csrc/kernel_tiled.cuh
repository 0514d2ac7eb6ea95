// kernel_tiled.cuh — shared-memory tiled backward induction for the 1-D inventory family
// (SDPB_COST_BACKORDER, lead_time 0: Recursion.java:129-161 with the lambdas of
// CLSPTesting.java:78-106 / CLSP.java:251-272).  Bit-identical to bi_generic by construction.
//
// Where the work goes.  Per (state x, action a, demand d_j) the reference computes
//     lvl = x + a - d_j;  c = ((fixed + v*a) + h*max(lvl,0)) + pi*max(-lvl,0)
//     Q += p_j * c;       Q += (p_j*gamma) * V_{t+1}(clamp(lvl))
// 1. One of the holding / penalty terms is always +0, so ((fv + hold) + pen) == fv + (hold + pen)
//    bit for bit, and (hold + pen) and the successor's value depend on the integer level
//    il = ix + ia - id_j alone.  Each CTA tabulates W[il] = (hold+pen, V_{t+1}[succ(il)]) for the
//    window of levels its tile can reach, once, in shared memory (coalesced fp64 loads of V_{t+1}).
// 2. A thread owns one order-up-to level y = x + a and R consecutive actions (so R states
//    x = y - a on a diagonal).  All R evaluations of a demand point share W[y - d_j] — ONE
//    16-byte shared-memory load — and the product (p_j*gamma)*V, leaving 4 fp64 instructions per
//    evaluation (+1/R): add, mul, add, add.  No FMA: Java has none.
// 3. The thread's R states do not change from one action chunk to the next, so the running
//    (best, argbest) per state stays in registers; a state's R residue classes live in R adjacent
//    threads and are merged once per launch through shared memory with the lexicographic
//    (value, action) rule == the reference's ascending first-wins scan (Recursion.java:146-157).
// 4. Small grids (C1: 1,001 states) cannot fill 148 SMs with state tiles alone, so the action
//    range is also split across CTAs (gridDim.y); the last CTA of a tile to finish merges the
//    partial optima.  Still one launch per period.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <string>
#include <vector>

#include "dev_model.cuh"

namespace sdpb {

constexpr int kTiledThreads = 256;
constexpr int kTiledR = 8;                                // actions (and states) per thread
constexpr int kTiledBX = kTiledThreads - kTiledR + 1;     // states per tile (249)

// bytes before the demand table: the level window, later aliased by the residue-merge area
__host__ __device__ inline size_t tiled_head_bytes(int WN) {
    const size_t w_bytes = (size_t)WN * 16;
    const size_t red_bytes = (((size_t)kTiledR * kTiledBX * 12) + 15) & ~(size_t)15;
    return w_bytes > red_bytes ? w_bytes : red_bytes;
}

struct TiledPeriod {
    bool ok = false;
    bool consec = false;  // demand indices are di_0, di_0+1, ...
    int di_max = 0, span = 0;
    int WN = 0;           // window entries
    size_t smem = 0;
    bool ok2 = false;     // bi_inv_tiled2 (needs consecutive demands)
    int WN2 = 0;
    size_t smem2 = 0;
};

struct TiledPlan {
    bool available = false;
    const char* why_not = "";
    std::vector<TiledPeriod> period;  // [T]
    int n_chunks = 0;                 // ceil(n_actions / R)
    int n_chunks2 = 0;                // ceil(n_actions / RA) for bi_inv_tiled2
    int variant = 0;                  // 0 = choose by size, 1 = bi_inv_tiled only, 2 = bi_inv_tiled2 when possible
    int sm_count = 148;
    int batch = 1;                    // instances solved side by side (sdpb_solve_batch): each gets 1/batch of the GPU,
                                      // so the action range is split only as far as THAT share needs
    // cross-CTA merge scratch for action splitting (allocated lazily by the owner)
    double* part_v = nullptr;
    int* part_a = nullptr;
    unsigned* counters = nullptr;
    size_t part_cap = 0, counter_cap = 0;
};

struct TiledArgs {
    int t, D, pmf_off;
    const double* Vn;
    double* Vt;
    int* Qt;
    long long lo, hi;
    int di_max, WN, n_chunks, chunks_per_split, nsplit;
    double* part_v;
    int* part_a;
    unsigned* counters;
};

template <bool IS_MIN, bool LAST, bool CONSEC>
__global__ void __launch_bounds__(kTiledThreads)
bi_inv_tiled(const __grid_constant__ DevModel M, const __grid_constant__ TiledArgs a) {
    constexpr int R = kTiledR, BX = kTiledBX, NT = kTiledThreads;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: [ W window | reduction area (aliased) ] [ (p, p*gamma) per demand ] [ e_j ]
    double2* W = reinterpret_cast<double2*>(smem_raw);
    const size_t head = tiled_head_bytes(a.WN);
    double2* PP = reinterpret_cast<double2*>(smem_raw + head);
    int* E = reinterpret_cast<int*>(smem_raw + head + (size_t)a.D * sizeof(double2));

    const int u = threadIdx.x;
    const long long X0 = a.lo + (long long)blockIdx.x * BX;  // first state of the tile
    const int split = blockIdx.y;

    // ---- stage the demand table ----
    for (int j = u; j < a.D; j += NT) {
        PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
        E[j] = a.di_max - M.pmf_di[a.pmf_off + j];
    }
    // ---- stage the level window: W[wi] <-> level index il = X0 - di_max + wi ----
    const bool lost = (M.flags & SDPB_F_LOST_SALES) != 0;
    for (int wi = u; wi < a.WN; wi += NT) {
        const long long il = X0 - a.di_max + wi;
        const double lvl = M.inv_min + (double)il * M.step;  // exact on the validated grid
        const double hold = M.h * fmax(lvl, 0.0);
        const double pen = M.pen * fmax(-lvl, 0.0);
        double vn = 0.0;
        if (!LAST) {
            long long is = il;
            if (lost) is = is > M.i_zero ? is : M.i_zero;
            is = is < M.nI - 1 ? is : M.nI - 1;  // upper clamp first (CLSPTesting.java:91-92)
            is = is > 0 ? is : 0;
            vn = a.Vn[is];
        }
        W[wi] = make_double2(hold + pen, vn);
    }
    __syncthreads();

    double best[R];
    int arg[R];
#pragma unroll
    for (int r = 0; r < R; r++) { best[r] = IS_MIN ? DBL_MAX : -DBL_MAX; arg[r] = kNoAction; }

    const double v = M.v_t[a.t - 1];
    const int c_begin = split * a.chunks_per_split;
    const int c_end = min(a.n_chunks, c_begin + a.chunks_per_split);
    const int e0 = a.D - 1;  // CONSEC: e_j = (D-1) - j

    // A thread whose R states X0 + u - r all lie beyond the block has nothing to evaluate: in the ragged last tile
    // (C2: 2001 states = 8 tiles of 249 + 9 states) seven of the eight warps skip the loop and leave their issue
    // slots to the other CTAs of the SM -- 10 % of a batch of such solves.
    const bool has_state = X0 + u - (R - 1) < a.hi;
    for (int c = has_state ? c_begin : c_end; c < c_end; c++) {
        double fv[R], acc[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int i = c * R + r;
            const double av = (double)i * M.step;
            const double fixedCost = av > 0.0 ? M.K : 0.0;
            fv[r] = fixedCost + v * av;  // fixedCost + variableCost (CLSPTesting.java:98-99,104)
            acc[r] = 0.0;
        }
        const double2* Wt = W + u + c * R;
#pragma unroll 4
        for (int j = 0; j < a.D; j++) {
            const double2 pp = PP[j];
            const double2 w = Wt[CONSEC ? (e0 - j) : E[j]];
            if (!LAST) {
                const double pv = pp.y * w.y;            // (p*gamma) * V_{t+1}(f)   Recursion.java:142
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const double cst = fv[r] + w.x;      // immediate value
                    acc[r] += pp.x * cst;                // Recursion.java:139
                    acc[r] += pv;
                }
            } else {
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const double cst = fv[r] + w.x;
                    acc[r] += pp.x * cst;
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int i = c * R + r;
            if (i <= M.max_order_idx && (IS_MIN ? (acc[r] < best[r]) : (acc[r] > best[r]))) {
                best[r] = acc[r];
                arg[r] = i;
            }
        }
    }

    // ---- merge the R residue classes of each state (aliases the window) ----
    __syncthreads();
    double* red_v = reinterpret_cast<double*>(smem_raw);
    int* red_a = reinterpret_cast<int*>(smem_raw + (size_t)R * BX * sizeof(double));
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int s = u - r;  // thread u, residue r evaluated state X0 + u - r
        if (s >= 0 && s < BX) { red_v[r * BX + s] = best[r]; red_a[r * BX + s] = arg[r]; }
    }
    __syncthreads();
    double bv = IS_MIN ? DBL_MAX : -DBL_MAX;
    int ba = kNoAction;
    const bool owner = u < BX && X0 + u < a.hi;
    if (u < BX) {
#pragma unroll
        for (int r = 0; r < R; r++) {
            const double ov = red_v[r * BX + u];
            const int oa = red_a[r * BX + u];
            if (better<IS_MIN>(ov, oa, bv, ba)) { bv = ov; ba = oa; }
        }
    }
    if (a.nsplit == 1) {
        if (owner) { a.Vt[X0 + u] = bv; a.Qt[X0 + u] = ba == kNoAction ? -1 : ba; }
        return;
    }
    // ---- action range was split over gridDim.y CTAs: the last one to arrive merges ----
    const size_t slot = ((size_t)blockIdx.x * a.nsplit + split) * BX + u;
    if (u < BX) { a.part_v[slot] = bv; a.part_a[slot] = ba; }
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (u == 0) is_last = (atomicAdd(&a.counters[blockIdx.x], 1u) == (unsigned)a.nsplit - 1u);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (owner) {
        bv = IS_MIN ? DBL_MAX : -DBL_MAX;
        ba = kNoAction;
        for (int sp = 0; sp < a.nsplit; sp++) {
            const size_t q = ((size_t)blockIdx.x * a.nsplit + sp) * BX + u;
            const double ov = __ldcg(a.part_v + q);
            const int oa = __ldcg(a.part_a + q);
            if (better<IS_MIN>(ov, oa, bv, ba)) { bv = ov; ba = oa; }
        }
        a.Vt[X0 + u] = bv;
        a.Qt[X0 + u] = ba == kNoAction ? -1 : ba;
    }
    if (u == 0) a.counters[blockIdx.x] = 0;  // ready for the next launch
}

// ---------------------------------------------------------------------------------------------
// bi_inv_tiled2 — the same model, 2-D register tile.  A thread owns Y = 4 consecutive order-up-to
// levels y and RA = 4 consecutive actions, i.e. 16 (state, action) pairs on 7 diagonals x = y - a.
// With consecutive integer demands the level y_k - d_j that slot k needs at demand j+1 is the one
// slot k-1 needed at demand j, so the immediate costs cst[k][r] = fv_r + W.x(level) and the
// successor values slide through registers: per demand point a thread loads ONE new level, forms 4
// new costs and 4 products (p*gamma)*V, and then spends 3 fp64 instructions on each of its 16
// evaluations (mul, add, add):  (4 + 4 + 48) / 16 = 3.5 per evaluation, 2.25 in the last period,
// against 4.125 / 3 in bi_inv_tiled.  The rotation is unrolled 4x so slots are compile-time
// registers.  The window is stored permuted ([level & 3][level >> 2]) so that the stride-4 level
// loads of a warp are unit-stride in shared memory.
__device__ __forceinline__ double2 lds_double2(unsigned shared_addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(shared_addr));
    return v;
}

constexpr int kT2Y = 4, kT2RA = 4;
constexpr int kT2BX = kTiledThreads * kT2Y - kT2RA + 1;  // 1021 states per tile

template <bool IS_MIN, bool LAST>
__global__ void __launch_bounds__(kTiledThreads, 2)
bi_inv_tiled2(const __grid_constant__ DevModel M, const __grid_constant__ TiledArgs a) {
    constexpr int Y = kT2Y, RA = kT2RA, BX = kT2BX, NT = kTiledThreads;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* W = reinterpret_cast<double2*>(smem_raw);  // permuted window, later aliased by the merge area
    const int Wq = (a.WN + 3) >> 2;
    const size_t head = (size_t)4 * Wq * sizeof(double2);
    double2* PP = reinterpret_cast<double2*>(smem_raw + head);

    const int u = threadIdx.x;
    const long long X0 = a.lo + (long long)blockIdx.x * BX;
    const int split = blockIdx.y;
    const int D = a.D;

    for (int j = u; j < D; j += NT) PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
    const bool lost = (M.flags & SDPB_F_LOST_SALES) != 0;
    for (int wi = u; wi < a.WN; wi += NT) {
        const long long il = X0 - a.di_max + wi;
        const double lvl = M.inv_min + (double)il * M.step;
        const double hold = M.h * fmax(lvl, 0.0);
        const double pen = M.pen * fmax(-lvl, 0.0);
        double vn = 0.0;
        if (!LAST) {
            long long is = il;
            if (lost) is = is > M.i_zero ? is : M.i_zero;
            is = is < M.nI - 1 ? is : M.nI - 1;
            is = is > 0 ? is : 0;
            vn = a.Vn[is];
        }
        W[(wi & 3) * Wq + (wi >> 2)] = make_double2(hold + pen, vn);
    }
    __syncthreads();

    const unsigned w_base = (unsigned)__cvta_generic_to_shared(W);
    const unsigned pp_base = (unsigned)__cvta_generic_to_shared(PP);

    // running optimum per diagonal delta = k - r in [-3, 3]  (state s = 4u + delta)
    double best[Y + RA - 1];
    int arg[Y + RA - 1];
#pragma unroll
    for (int q = 0; q < Y + RA - 1; q++) { best[q] = IS_MIN ? DBL_MAX : -DBL_MAX; arg[q] = kNoAction; }

    const double v = M.v_t[a.t - 1];
    const int c_begin = split * a.chunks_per_split;
    const int c_end = min(a.n_chunks, c_begin + a.chunks_per_split);

    const bool has_state = X0 + (long long)Y * u - (RA - 1) < a.hi;  // (see bi_inv_tiled: the ragged last tile)
    for (int c = has_state ? c_begin : c_end; c < c_end; c++) {
        double fv[RA], acc[Y][RA], cst[Y][RA], Vw[Y];
#pragma unroll
        for (int r = 0; r < RA; r++) {
            const double av = (double)(c * RA + r) * M.step;
            fv[r] = (av > 0.0 ? M.K : 0.0) + v * av;
        }
        // level needed by slot k at demand j:  wi = 4u + 4c + (D-1-j) + k
        int b = Y * u + RA * c + (D - 1);
#pragma unroll
        for (int k = 0; k < Y; k++) {
            const int wi = b + k;
            const double2 w = lds_double2(w_base + (unsigned)(((wi & 3) * Wq + (wi >> 2)) << 4));
#pragma unroll
            for (int r = 0; r < RA; r++) { cst[k][r] = fv[r] + w.x; acc[k][r] = 0.0; }
            Vw[k] = w.y;
        }
        // One demand point for all 16 pairs.  JJ is the rotation phase (j mod 4): level slot k lives in
        // physical register slot (k - JJ) & 3.  Software-pipelined: this step's (p, p*gamma) was loaded
        // one step ago; the loads for the next step (probabilities, the level entering slot 0) issue
        // first.  Shared memory is addressed through explicit 32-bit shared-space addresses so the
        // base is not re-derived every step.
#define SDPB_T2_STEP(JJ)                                                                         \
        {                                                                                            \
            const double2 pp = pp_next;                                                              \
            pp_next = lds_double2(pp_addr);                                                          \
            pp_addr += (j + 1 < D - 1) ? 16u : 0u;                                                   \
            const int wn = max(b - 1, 0);                                                            \
            const double2 wnew = lds_double2(w_base + (unsigned)(((wn & 3) * Wq + (wn >> 2)) << 4)); \
            _Pragma("unroll") for (int k = 0; k < Y; k++) {                                          \
                const int ph = (k - (JJ)) & 3;                                                       \
                if (!LAST) {                                                                         \
                    const double pv = pp.y * Vw[ph];                                                 \
                    _Pragma("unroll") for (int r = 0; r < RA; r++) {                                 \
                        acc[k][r] += pp.x * cst[ph][r];                                              \
                        acc[k][r] += pv;                                                             \
                    }                                                                                \
                } else {                                                                             \
                    _Pragma("unroll") for (int r = 0; r < RA; r++) acc[k][r] += pp.x * cst[ph][r];   \
                }                                                                                    \
            }                                                                                        \
            const int pn = (3 - (JJ)) & 3; /* freed slot becomes slot 0 of the next demand */        \
            _Pragma("unroll") for (int r = 0; r < RA; r++) cst[pn][r] = fv[r] + wnew.x;              \
            Vw[pn] = wnew.y;                                                                         \
            b -= 1;                                                                                  \
            j += 1;                                                                                  \
        }
        double2 pp_next = lds_double2(pp_base);
        unsigned pp_addr = pp_base + (D > 1 ? 16u : 0u);
        int j = 0;
        for (; j + 4 <= D;) { SDPB_T2_STEP(0) SDPB_T2_STEP(1) SDPB_T2_STEP(2) SDPB_T2_STEP(3) }
        if (j < D) SDPB_T2_STEP(0)
        if (j < D) SDPB_T2_STEP(1)
        if (j < D) SDPB_T2_STEP(2)
#undef SDPB_T2_STEP
        // ascending actions within the chunk, strict compare: first optimum wins
#pragma unroll
        for (int r = 0; r < RA; r++) {
            const int i = c * RA + r;
#pragma unroll
            for (int k = 0; k < Y; k++) {
                const int q = k - r + (RA - 1);
                if (i <= M.max_order_idx && (IS_MIN ? (acc[k][r] < best[q]) : (acc[k][r] > best[q]))) {
                    best[q] = acc[k][r];
                    arg[q] = i;
                }
            }
        }
    }

    // ---- merge: state s gets one partial from thread s/4 (delta >= 0) and one from thread s/4+1 ----
    __syncthreads();
    double* redA_v = reinterpret_cast<double*>(smem_raw);
    double* redB_v = redA_v + NT * Y;
    int* redA_a = reinterpret_cast<int*>(redB_v + NT * Y);
    int* redB_a = redA_a + NT * Y;
#pragma unroll
    for (int k = 0; k < Y; k++) { redB_v[Y * u + k] = IS_MIN ? DBL_MAX : -DBL_MAX; redB_a[Y * u + k] = kNoAction; }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < Y + RA - 1; q++) {
        const int delta = q - (RA - 1);
        const int s = Y * u + delta;
        if (delta >= 0) { redA_v[s] = best[q]; redA_a[s] = arg[q]; }
        else if (s >= 0) { redB_v[s] = best[q]; redB_a[s] = arg[q]; }
    }
    __syncthreads();
    // each thread finishes 4 states (s = u, u + NT, ...): coalesced writes
#pragma unroll
    for (int k = 0; k < Y; k++) {
        const int s = u + k * NT;
        if (s >= BX) continue;
        double bv = redA_v[s];
        int ba = redA_a[s];
        if (better<IS_MIN>(redB_v[s], redB_a[s], bv, ba)) { bv = redB_v[s]; ba = redB_a[s]; }
        if (a.nsplit == 1) {
            if (X0 + s < a.hi) { a.Vt[X0 + s] = bv; a.Qt[X0 + s] = ba == kNoAction ? -1 : ba; }
        } else {
            const size_t slot = ((size_t)blockIdx.x * a.nsplit + split) * BX + s;
            a.part_v[slot] = bv;
            a.part_a[slot] = ba;
        }
    }
    if (a.nsplit == 1) return;
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (u == 0) is_last = (atomicAdd(&a.counters[blockIdx.x], 1u) == (unsigned)a.nsplit - 1u);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
#pragma unroll
    for (int k = 0; k < Y; k++) {
        const int s = u + k * NT;
        if (s >= BX || X0 + s >= a.hi) continue;
        double bv = IS_MIN ? DBL_MAX : -DBL_MAX;
        int ba = kNoAction;
        for (int sp = 0; sp < a.nsplit; sp++) {
            const size_t q = ((size_t)blockIdx.x * a.nsplit + sp) * BX + s;
            const double ov = __ldcg(a.part_v + q);
            const int oa = __ldcg(a.part_a + q);
            if (better<IS_MIN>(ov, oa, bv, ba)) { bv = ov; ba = oa; }
        }
        a.Vt[X0 + s] = bv;
        a.Qt[X0 + s] = ba == kNoAction ? -1 : ba;
    }
    if (u == 0) a.counters[blockIdx.x] = 0;
}

// ---- host side --------------------------------------------------------------------------------
inline void plan_tiled(TiledPlan& P, const sdpb_model& m, const DevModel& d, const std::vector<int>& pmf_len,
                       const std::vector<int>& pmf_off, const std::vector<int>& pdi, bool /*dedup*/,
                       int sm_count) {
    P.available = false;
    P.sm_count = sm_count;
    if (m.cost_kind != SDPB_COST_BACKORDER) { P.why_not = "only the backorder cost kind is tiled"; return; }
    if (m.lead_time != 0) { P.why_not = "lead-time states are not tiled yet"; return; }
    if (!(m.flags & SDPB_F_CLAMP_INV)) { P.why_not = "needs the inventory clamp"; return; }
    P.n_chunks = (d.max_order_idx + 1 + kTiledR - 1) / kTiledR;
    P.period.assign(m.T, TiledPeriod{});
    bool any = false;
    for (int t = 0; t < m.T; t++) {
        TiledPeriod& tp = P.period[t];
        if ((m.flags & SDPB_F_GY_MODE) && t == 0) continue;  // the G(y) pass runs on the generic kernel
        const int D = pmf_len[t];
        const int* di = pdi.data() + pmf_off[t];
        int lo = di[0], hi = di[0];
        bool consec = true;
        for (int j = 0; j < D; j++) {
            lo = std::min(lo, di[j]);
            hi = std::max(hi, di[j]);
            if (di[j] != di[0] + j) consec = false;
        }
        tp.consec = consec;
        tp.di_max = hi;
        tp.span = hi - lo;
        tp.WN = kTiledBX + P.n_chunks * kTiledR + tp.span;
        tp.smem = tiled_head_bytes(tp.WN) + (size_t)D * 16 + (size_t)D * 4 + 16;
        tp.ok = tp.smem <= 200 * 1024;
        any = any || tp.ok;
        // 2-D register tile variant
        P.n_chunks2 = (d.max_order_idx + 1 + kT2RA - 1) / kT2RA;
        tp.WN2 = kTiledThreads * kT2Y + P.n_chunks2 * kT2RA + D;
        const size_t head2 = (size_t)4 * ((tp.WN2 + 3) >> 2) * 16;
        const size_t red2 = (size_t)kTiledThreads * kT2Y * 2 * 12;
        tp.smem2 = std::max(head2, red2) + (size_t)D * 16 + 16;
        tp.ok2 = consec && tp.smem2 <= 100 * 1024;
    }
    if (!any) { P.why_not = "no period qualifies (G(y) pass only, or the level window does not fit in shared memory)"; return; }
    P.available = true;
}

template <bool IS_MIN, bool LAST, bool CONSEC>
inline cudaError_t launch_tiled_inst(const DevModel& dm, const TiledArgs& a, dim3 grid, size_t smem,
                                     cudaStream_t stream) {
    auto k = bi_inv_tiled<IS_MIN, LAST, CONSEC>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    k<<<grid, kTiledThreads, smem, stream>>>(dm, a);
    return cudaGetLastError();
}

inline int tiled_scratch(TiledPlan& P, long long tiles, int nsplit, int bx, cudaStream_t stream) {
    if (nsplit <= 1) return SDPB_OK;
    const size_t need = (size_t)tiles * nsplit * bx;
    if (need > P.part_cap) {
        if (P.part_v) cudaFree(P.part_v);
        if (P.part_a) cudaFree(P.part_a);
        P.part_v = nullptr; P.part_a = nullptr; P.part_cap = 0;
        if (cudaMalloc((void**)&P.part_v, need * sizeof(double)) != cudaSuccess) return SDPB_ERR_NOMEM;
        if (cudaMalloc((void**)&P.part_a, need * sizeof(int)) != cudaSuccess) return SDPB_ERR_NOMEM;
        P.part_cap = need;
    }
    if ((size_t)tiles > P.counter_cap) {
        if (P.counters) cudaFree(P.counters);
        P.counters = nullptr; P.counter_cap = 0;
        if (cudaMalloc((void**)&P.counters, (size_t)tiles * sizeof(unsigned)) != cudaSuccess) return SDPB_ERR_NOMEM;
        if (cudaMemsetAsync(P.counters, 0, (size_t)tiles * sizeof(unsigned), stream) != cudaSuccess) return SDPB_ERR_CUDA;
        P.counter_cap = (size_t)tiles;
    }
    return SDPB_OK;
}

template <bool IS_MIN, bool LAST>
inline cudaError_t launch_tiled2_inst(const DevModel& dm, const TiledArgs& a, dim3 grid, size_t smem,
                                      cudaStream_t stream) {
    auto k = bi_inv_tiled2<IS_MIN, LAST>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    k<<<grid, kTiledThreads, smem, stream>>>(dm, a);
    return cudaGetLastError();
}

// For a period whose plan has tp.ok or tp.ok2.  Returns SDPB_OK, SDPB_ERR_CUDA or SDPB_ERR_NOMEM.
// *variant_used: 1 = bi_inv_tiled, 2 = bi_inv_tiled2.
inline int launch_tiled(TiledPlan& P, const DevModel& dm, int t, int D, int pmf_off, const double* Vn,
                        double* Vt, int* Qt, long long lo, long long hi, cudaStream_t stream, int* variant_used) {
    const TiledPeriod& tp = P.period[t - 1];
    const long long n = hi - lo;
    if (n <= 0) return SDPB_OK;
    const bool last = (Vn == nullptr);  // period T without a terminal table (Recursion.java:140)
    const bool mn = dm.is_min != 0;
    const long long target = std::max(1LL, 4LL * P.sm_count / P.batch);  // about 4 CTAs per SM (of this instance's share)
    TiledArgs a;
    a.t = t; a.D = D; a.pmf_off = pmf_off; a.Vn = Vn; a.Vt = Vt; a.Qt = Qt; a.lo = lo; a.hi = hi;
    a.di_max = tp.di_max;

    // the 2-D register tile pays off once there are enough 1021-state tiles to fill the machine
    const long long tiles2 = (n + kT2BX - 1) / kT2BX;
    // measured on C5 (200 x 200): the 2-D register tile (with its action split) wins from ~64 tiles on
    // (S = 1e5: 3.36 vs 4.02 ms, 2e5: 6.8 vs 8.0, 3e5: 9.0 vs 11.9) and is level at 3e4 (1.40 vs 1.37)
    // (a batch fills the machine with its instances: 64 C2 solves 3.62 ms on bi_inv_tiled, 3.06 ms on this one)
    const bool use2 = tp.ok2 && (P.variant == 2 || (P.variant == 0 && tiles2 * P.batch >= 64) || !tp.ok);
    if (use2) {
        int nsplit = 1;
        // enough CTAs for ~8 waves of 2 CTAs per SM: a grid of a few waves loses its last, partial one
        // (measured, C5: S = 1e6 32.9 -> 30.0 ms, S = 1e5 3.36 -> 3.17 ms; no change at 3e5 and 3e6)
        // (one instance of a batch: 3 waves of its share -- measured 64 x C2: 8 waves 3.15 ms, 4: 3.08, 3: 3.06, 1: 3.26)
        const long long want = P.batch > 1 ? std::max(1LL, 6LL * P.sm_count / P.batch) : 16LL * P.sm_count;
        if (tiles2 < want) nsplit = (int)std::min<long long>(P.n_chunks2, (want + tiles2 - 1) / tiles2);
        const int cps = (P.n_chunks2 + nsplit - 1) / nsplit;
        nsplit = (P.n_chunks2 + cps - 1) / cps;
        int rc = tiled_scratch(P, tiles2, nsplit, kT2BX, stream);
        if (rc != SDPB_OK) return rc;
        a.WN = tp.WN2; a.n_chunks = P.n_chunks2; a.chunks_per_split = cps; a.nsplit = nsplit;
        a.part_v = P.part_v; a.part_a = P.part_a; a.counters = P.counters;
        const dim3 grid((unsigned)tiles2, (unsigned)nsplit);
        cudaError_t e;
        if (mn) e = last ? launch_tiled2_inst<true, true>(dm, a, grid, tp.smem2, stream)
                         : launch_tiled2_inst<true, false>(dm, a, grid, tp.smem2, stream);
        else e = last ? launch_tiled2_inst<false, true>(dm, a, grid, tp.smem2, stream)
                      : launch_tiled2_inst<false, false>(dm, a, grid, tp.smem2, stream);
        if (e != cudaSuccess) return SDPB_ERR_CUDA;
        *variant_used = 2;
        return SDPB_OK;
    }

    const long long tiles = (n + kTiledBX - 1) / kTiledBX;
    // split the action range when state tiles are too few to fill the machine
    int nsplit = 1;
    if (tiles < target) nsplit = (int)std::min<long long>(P.n_chunks, (target + tiles - 1) / tiles);
    const int cps = (P.n_chunks + nsplit - 1) / nsplit;
    nsplit = (P.n_chunks + cps - 1) / cps;
    int rc = tiled_scratch(P, tiles, nsplit, kTiledBX, stream);
    if (rc != SDPB_OK) return rc;
    a.WN = tp.WN; a.n_chunks = P.n_chunks; a.chunks_per_split = cps; a.nsplit = nsplit;
    a.part_v = P.part_v; a.part_a = P.part_a; a.counters = P.counters;
    const dim3 grid((unsigned)tiles, (unsigned)nsplit);
    cudaError_t e;
#define SDPB_TILED_CASE(MN, LS, CS) e = launch_tiled_inst<MN, LS, CS>(dm, a, grid, tp.smem, stream)
    if (mn) {
        if (last) { if (tp.consec) SDPB_TILED_CASE(true, true, true); else SDPB_TILED_CASE(true, true, false); }
        else      { if (tp.consec) SDPB_TILED_CASE(true, false, true); else SDPB_TILED_CASE(true, false, false); }
    } else {
        if (last) { if (tp.consec) SDPB_TILED_CASE(false, true, true); else SDPB_TILED_CASE(false, true, false); }
        else      { if (tp.consec) SDPB_TILED_CASE(false, false, true); else SDPB_TILED_CASE(false, false, false); }
    }
#undef SDPB_TILED_CASE
    if (e != cudaSuccess) return SDPB_ERR_CUDA;
    *variant_used = 1;
    return SDPB_OK;
}

inline void free_tiled(TiledPlan& P) {
    if (P.part_v) cudaFree(P.part_v);
    if (P.part_a) cudaFree(P.part_a);
    if (P.counters) cudaFree(P.counters);
    P.part_v = nullptr; P.part_a = nullptr; P.counters = nullptr;
}

}  // namespace sdpb
