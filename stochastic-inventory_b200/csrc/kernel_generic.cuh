// kernel_generic.cuh — the general backward-induction kernel: one launch per period, every
// (state, action, demand) triple evaluated exactly as the reference's lambdas write it.
//
//   bi_generic<KIND, SURVIVAL, IS_MIN, G>
//     G lanes cooperate on one state.  G = 32 for the backorder kinds (lanes stride over the
//     actions, so the V_{t+1} gather V[(x+a-d, .., a)] is unit-stride across lanes, then a
//     warp-shuffle (value, action) reduction picks the optimum).  G = 1 for the cash kinds (one
//     thread per state with the cash axis innermost, so lanes of a warp hold consecutive cash
//     levels and gather consecutive V[(x', w')] addresses; actions run serially in the thread
//     because |A(s)| depends on the cash level).
//   reach_forward<KIND>
//     forward reachability through every feasible action and demand — the set of states the
//     reference's top-down memoisation visits (Recursion.java:89-90,141-142) — used to reproduce
//     getOptTable()/getCacheActions() row sets (Recursion.java:169-186).
//
// Reference loops restated (relative to /root/reference):
//   src/sdp/inventory/Recursion.java:129-161        src/sdp/cash/CashRecursion.java:98-138
//   src/sdp/inventory/LeadtimeRecursion.java:49-73  src/sdp/cash/CashLeadtimeRecursion.java:50-77
//   src/sdp/cash/CashRecursionXR.java:82-124        src/sdp/cash/RiskRecursion.java:66-104
// and the lambdas named in include/sdpb200.h.  Per-(s,a) sub-expressions that do not depend on
// the demand are hoisted out of the j loop; hoisting does not change any rounding.
#pragma once
#include "dev_model.cuh"

namespace sdpb {

// A decoded state plus everything that is constant over its (a, d) loop.
struct StateCtx {
    int t;
    int ix, iq1, iq2, iw;
    double x, q1, w;  // w: cash (R for the XR kind)
    int nA;           // |A(s)|
    bool capped;      // XR kind: the order-up-to range of CashConstraintXR.java:71-75 is longer than max_order_idx + 1
    double price, v, ovh;
    bool last, lost, gy;
    long long strideX;
};

// Per-(s,a) invariants.
struct ActionCtx {
    double a;
    double stock;     // x + a, x + preQ, or the order-up-to level
    int iy;           // grid index of `stock` relative to inv_min
    double fv;        // backorder: fixedCost + variableCost
    double initCash;  // w, or R - v*x for XR
    double deposite;  // CASH_DEPOSIT / XR
    double before_minus_interest;  // CASH_OVERDRAFT: cashBalanceBefore - interest
    double fixedCost, variableCost;  // kinds whose balance depends on the demand keep them separate
    long long pipe;   // successor's pipeline-slot offset
};

// |A(s)| (S.nA, S.capped) of a state whose t, x, w, v and last are set; shared by the grid kernels and the
// top-down engine (topdown.cu), whose states are not grid points.
template <int KIND>
__device__ __forceinline__ void feasible_actions(const DevModel& M, StateCtx& S) {
    int nA = M.max_order_idx + 1;
    S.capped = false;
    if (KIND == SDPB_COST_CASH_XR) {
        // CashConstraintXR.java:71-75
        const double rv = S.w / S.v;
        const double maxY = rv < S.x ? S.x : rv;
        const int length = (int)(maxY - S.x) + 1;
        S.capped = length > nA;  // dense-grid artefact: the reference has no cap (sdpb_reach reports it)
        nA = length < nA ? length : nA;
    } else {
        if (M.flags & SDPB_F_CASH_LIMITED_ACTIONS) {
            // CashConstraint.java:96-99, cashSurvival.java:103-110
            const double bound = fmax(0.0, ((S.w - M.reserve_t[S.t - 1]) - M.reserve2) / S.v);
            nA = (int)fmin((double)M.max_order_idx, bound) + 1;
        }
        if ((M.flags & SDPB_F_NO_ORDER_LAST) && S.last) nA = 1;
    }
    S.nA = nA;
}

// `dedup`: idx addresses a VIRTUAL state (y = x + preQ, [preQ2], [cash]) with preQ folded into the
// inventory index — lead-time models depend on (x, preQ) only through their sum, so every real
// state with the same sum has the same value and policy (exactly, not approximately).
template <int KIND>
__device__ __forceinline__ StateCtx decode_state(const DevModel& M, int t, long long idx, bool dedup = false) {
    StateCtx S;
    long long r = idx;
    S.t = t;
    S.iw = 0; S.iq1 = 0; S.iq2 = 0;
    if (KIND != SDPB_COST_BACKORDER) { S.iw = (int)(r % M.nW); r /= M.nW; }
    if (M.lead >= 2) { S.iq2 = (int)(r % M.nQ); r /= M.nQ; }
    if (M.lead >= 1 && !dedup) { S.iq1 = (int)(r % M.nQ); r /= M.nQ; }
    S.ix = (int)r;
    S.x = M.inv_min + (double)S.ix * M.step;
    S.q1 = (double)S.iq1 * M.step;
    S.w = 0.0;
    if (KIND != SDPB_COST_BACKORDER) {
        const long long k = M.kmin + S.iw;
        S.w = (KIND != SDPB_COST_CASH_XR && M.quantiser == SDPB_Q_DIV) ? (double)k / M.q_div : (double)k;
    }
    S.last = (t == M.T);
    S.price = M.price_t[t - 1];
    S.v = M.v_t[t - 1];
    S.ovh = M.ovh_t[t - 1];
    S.lost = (M.flags & SDPB_F_LOST_SALES) != 0;
    S.gy = (KIND == SDPB_COST_BACKORDER) && (M.flags & SDPB_F_GY_MODE) && t == 1;
    S.strideX = (long long)M.nW * (M.lead >= 1 ? M.nQ : 1) * (M.lead >= 2 ? M.nQ : 1);
    feasible_actions<KIND>(M, S);
    return S;
}

template <int KIND>
__device__ __forceinline__ ActionCtx prep_action(const DevModel& M, const StateCtx& S, int i) {
    ActionCtx A;
    A.a = (double)i * M.step;
    A.pipe = 0;
    if (M.lead == 1) A.pipe = (long long)i * M.nW;
    if (M.lead == 2) A.pipe = ((long long)S.iq2 * M.nQ + i) * M.nW;
    A.fv = 0.0; A.deposite = 0.0; A.before_minus_interest = 0.0; A.initCash = S.w;
    A.fixedCost = 0.0; A.variableCost = 0.0;
    if (KIND == SDPB_COST_BACKORDER) {
        // CLSPTesting.java:96-106 / Leadtime.java:71-81 / CLSPforDraw.java:156-170
        const double fixedCost = S.gy ? 0.0 : (A.a > 0.0 ? M.K : 0.0);
        const double variableCost = S.gy ? S.v * S.x : S.v * A.a;
        A.fv = fixedCost + variableCost;
        A.stock = S.gy ? S.x : (M.lead > 0 ? S.x + S.q1 : S.x + A.a);
        A.iy = S.gy ? S.ix : (M.lead > 0 ? S.ix + S.iq1 : S.ix + i);
        return A;
    }
    double fixedCost, variableCost;
    if (KIND == SDPB_COST_CASH_XR) {
        // CashConstraintXR.java:78-86: the action is the order-up-to level y = x + i*step
        A.stock = S.x + A.a;
        A.iy = S.ix + i;
        const double act = A.stock - S.x;
        fixedCost = A.stock > S.x ? M.K : 0.0;
        variableCost = S.v * act;
        A.initCash = S.w - S.v * S.x;
    } else {
        A.stock = M.lead > 0 ? S.x + S.q1 : S.x + A.a;
        A.iy = M.lead > 0 ? S.ix + S.iq1 : S.ix + i;
        fixedCost = A.a > 0.0 ? M.K : 0.0;
        variableCost = S.v * A.a;
    }
    A.fixedCost = fixedCost;
    A.variableCost = variableCost;
    if (KIND == SDPB_COST_CASH_OD_LIMIT || KIND == SDPB_COST_CASH_OD_TESTING || KIND == SDPB_COST_CASH_LOAN)
        return A;  // their balances depend on the demand: nothing more to hoist
    if (KIND == SDPB_COST_CASH_OVERDRAFT) {
        // CashOverdraft.java:85-95
        const double before = ((A.initCash - fixedCost) - variableCost) - S.ovh;
        double interest;
        if (before >= 0.0)
            interest = M.neg_r0 * before;
        else if (before >= -M.interest_free)
            interest = 0.0;
        else if (before >= -M.od_limit)
            interest = M.r2 * (-before - M.interest_free);
        else
            interest = M.r3 * (-before - M.od_limit) + M.r2_limit_term;
        A.before_minus_interest = before - interest;
    } else {
        A.deposite = ((A.initCash - fixedCost) - variableCost) * M.one_plus_dr;
    }
    return A;
}

// Math.max(x, 0) / Math.min(a, b) for the values that occur here (no NaN; a zero result is +0.0 either way):
// a compare and a select instead of fmax/fmin's NaN-propagating sequence (10 instructions per call in SASS).
__device__ __forceinline__ double jmax0(double x) { return x > 0.0 ? x : 0.0; }
__device__ __forceinline__ double jmin(double a, double b) { return a < b ? a : b; }

// Immediate value c(s,a,d).  `after` receives the end-of-period cash balance for the one kind whose
// transition uses it directly instead of w + c (CashOverdraftTesting.java:103-111).
template <int KIND>
__device__ __forceinline__ double immediate(const DevModel& M, const StateCtx& S, const ActionCtx& A,
                                            double d, double& after) {
    const double lvl = A.stock - d;
    after = 0.0;
    if (KIND == SDPB_COST_BACKORDER) {
        const double hold = M.h * jmax0(lvl);
        const double pen = M.pen * jmax0(-lvl);
        return (A.fv + hold) + pen;
    }
    const double revenue = S.price * jmin(A.stock, d);
    if (KIND == SDPB_COST_CASH_OD_LIMIT) {
        // CashOverdraftLimit.java:70-86
        const double hold = M.h * jmax0(lvl);
        const double before = (((S.w - A.fixedCost) - A.variableCost) - hold) - S.ovh;
        const double interest = M.r2 * jmax0(-before);
        const double deposite = M.dr * jmax0(before);
        const double bal = ((before - interest) + deposite) + revenue;
        double inc = bal - S.w;
        inc += S.last ? M.salvage * jmax0(lvl) : 0.0;
        return inc;
    }
    if (KIND == SDPB_COST_CASH_OD_TESTING) {
        // CashOverdraftTesting.java:85-99 (and :103-111 for the balance the transition keeps)
        const double hold = M.h * jmax0(lvl);
        const double before = (((S.w + revenue) - A.fixedCost) - A.variableCost) - hold;
        const double interest = M.r2 * jmax0(-before);
        after = before - interest;
        return after - S.w;
    }
    if (KIND == SDPB_COST_CASH_LOAN) {
        // TestPaper.java:82-93
        const double hold = S.last ? 0.0 : M.h * jmax0(lvl);
        const double deposites = M.dr * jmax0(S.w - A.variableCost);
        const double loanPayed = M.r2 * jmax0(A.variableCost - S.w);
        double inc = (((revenue - A.variableCost) - hold) + deposites) - loanPayed;
        inc += S.last ? M.salvage * jmax0(lvl) : 0.0;
        return inc;
    }
    double inc;
    if (KIND == SDPB_COST_CASH_OVERDRAFT) {
        const double after = A.before_minus_interest + revenue;  // CashOverdraft.java:99
        inc = after - A.initCash;
    } else {
        const double hold = M.h * jmax0(lvl);
        inc = (((M.one_minus_rho * revenue + A.deposite) - hold) - S.ovh) - A.initCash;
    }
    const double sal = S.last ? M.salvage * jmax0(lvl) : 0.0;
    inc += sal;
    if (KIND == SDPB_COST_CASH_DEPOSIT) {
        const double endCash = A.initCash + inc;  // CashConstraint.java:116-119
        if (endCash < 0.0) inc += M.pen * endCash;
    }
    return inc;
}

// Successor f(s,a,d) as a flattened grid index; `bankrupt` = successor cash < 0 (survival only).
template <int KIND>
__device__ __forceinline__ long long successor(const DevModel& M, const StateCtx& S, const ActionCtx& A,
                                               int di, double c, double after, bool& bankrupt) {
    int il = A.iy - di;
    if (S.lost) il = max(il, M.i_zero);
    il = min(il, M.nI - 1);  // upper clamp first, then lower (CLSPTesting.java:91-92)
    il = max(il, 0);
    bankrupt = false;
    if (KIND == SDPB_COST_BACKORDER) return il * S.strideX + A.pipe;
    // CashConstraint.java:123-133 / CashConstraintXR.java:95-110
    double nw = (KIND == SDPB_COST_CASH_OD_TESTING) ? after : A.initCash + c;
    nw = nw > M.cash_max ? M.cash_max : nw;
    nw = nw < M.cash_min ? M.cash_min : nw;
    long long kk, k;
    if (M.quantiser == SDPB_Q_TRUNC) {
        // TestPaper.java:107-109: round from period q_from_period on, then (int) truncation
        if (M.q_from_period > 0 && S.t >= M.q_from_period) nw = (double)jround(nw * M.q_mul) / M.q_div;
        kk = k = (long long)nw;
    } else {
        kk = jround(nw * M.q_mul);
        // Java long division; q_idiv == 1 (round(w*1)/1) is the common case and needs no divide
        k = (M.quantiser == SDPB_Q_DIV || M.q_idiv == 1) ? kk : jdiv(kk, M.q_idiv, M.q_magic);
    }
    bankrupt = k < 0;  // quantised cash < 0 (q_div > 0)
    if (KIND == SDPB_COST_CASH_XR) {
        const double nwq = (M.quantiser == SDPB_Q_DIV) ? (double)kk / M.q_div : (double)k;
        const double nx = M.inv_min + (double)il * M.step;
        k = jround(nwq + S.v * nx);  // nextR, CashConstraintXR.java:107
    }
    long long kw = k - M.kmin;
    kw = kw < 0 ? 0 : (kw >= M.nW ? M.nW - 1 : kw);
    return il * S.strideX + A.pipe + kw;
}

// What the dense grid did to the successor that the reference's lambdas would not have done:
// bit 0: the inventory level left [inv_min, inv_max] although the model does not clamp (Leadtime.java:65-66) and
//        was folded onto the boundary row;  bit 1: the cash balance was clamped at cash_min / cash_max (part of
//        the reference lambdas, CashConstraint.java:128-129; reported only on request).  Used by reach_forward.
template <int KIND>
__device__ __forceinline__ unsigned successor_clip(const DevModel& M, const StateCtx& S, const ActionCtx& A, int di,
                                                   double c, double after) {
    unsigned r = 0;
    int il = A.iy - di;
    if (S.lost) il = max(il, M.i_zero);
    if (!(M.flags & SDPB_F_CLAMP_INV) && (il < 0 || il > M.nI - 1)) r |= 1u;
    if (KIND != SDPB_COST_BACKORDER) {
        const double nw = (KIND == SDPB_COST_CASH_OD_TESTING) ? after : A.initCash + c;
        if (nw > M.cash_max || nw < M.cash_min) r |= 2u;
    }
    return r;
}

// successor() in 32-bit integer arithmetic for DevModel::small grids (identical results: every quantity is
// below 2^31 there, checked on the host).
template <int KIND>
__device__ __forceinline__ int successor32(const DevModel& M, const StateCtx& S, const ActionCtx& A, int di, double c,
                                           double after, bool& bankrupt) {
    int il = A.iy - di;
    if (S.lost) il = max(il, M.i_zero);
    il = min(il, M.nI - 1);
    il = max(il, 0);
    bankrupt = false;
    const int strideX = (int)S.strideX, pipe = (int)A.pipe;
    if (KIND == SDPB_COST_BACKORDER) return il * strideX + pipe;
    double nw = (KIND == SDPB_COST_CASH_OD_TESTING) ? after : A.initCash + c;
    nw = nw > M.cash_max ? M.cash_max : nw;
    nw = nw < M.cash_min ? M.cash_min : nw;
    int kk, k;
    if (M.quantiser == SDPB_Q_TRUNC) {
        if (M.q_from_period > 0 && S.t >= M.q_from_period) nw = (double)jround32(nw * M.q_mul) / M.q_div;
        kk = k = (int)nw;
    } else {
        kk = jround32(nw * M.q_mul);
        k = (M.quantiser == SDPB_Q_DIV || M.q_idiv == 1) ? kk : jdiv32(kk, (int)M.q_idiv, M.q_magic);
    }
    bankrupt = k < 0;
    if (KIND == SDPB_COST_CASH_XR) {
        const double nwq = (M.quantiser == SDPB_Q_DIV) ? (double)kk / M.q_div : (double)k;
        const double nx = M.inv_min + (double)il * M.step;
        k = jround32(nwq + S.v * nx);
    }
    int kw = k - (int)M.kmin;
    kw = max(min(kw, M.nW - 1), 0);
    return il * strideX + pipe + kw;
}

// DEDUP: [lo, hi) indexes virtual states and (Vt, Qt) are the virtual tables H; see expand_dedup.
template <int KIND, bool SURVIVAL, bool IS_MIN, int G, bool DEDUP>
__global__ void __launch_bounds__(256)
bi_generic(const __grid_constant__ DevModel M, const int t, const int D, const int pmf_off,
           const double* __restrict__ Vn, double* __restrict__ Vt, int* __restrict__ Qt,
           const long long lo, const long long hi) {
    const long long gid = (long long)blockIdx.x * (256 / G) + threadIdx.x / G;
    const int lane = threadIdx.x % G;
    const long long idx = lo + gid;
    const bool live = idx < hi;  // dead groups still take part in the shuffles below
    const StateCtx S = decode_state<KIND>(M, t, live ? idx : lo, DEDUP);

    double best = IS_MIN ? DBL_MAX : -DBL_MAX;
    int besti = kNoAction;

    const bool small = M.small != 0;
    const double2* __restrict__ rec = M.pmf_rec + 2 * (size_t)pmf_off;  // (d, p), (p*gamma, d/step) per demand point
    for (int i = lane; i < S.nA; i += G) {
        const ActionCtx A = prep_action<KIND>(M, S, i);
        double acc = 0.0;
        if (Vn == nullptr) {  // period T of an engine without a boundary function (Recursion.java:140)
            for (int j = 0; j < D; j++) {
                double after;
                const double2 dp = __ldg(rec + 2 * j);
                const double c = immediate<KIND>(M, S, A, dp.x, after);
                if (!SURVIVAL) acc += dp.y * c;                           // Recursion.java:139
                if (SURVIVAL) {                                           // RiskRecursion.java:80-84
                    const double finalCash = A.initCash + c;
                    acc += dp.y * (finalCash >= 0.0 ? 1.0 : 0.0);
                }
            }
        } else if (small) {
#pragma unroll 2
            for (int j = 0; j < D; j++) {
                double after;
                const double2 dp = __ldg(rec + 2 * j), gi = __ldg(rec + 2 * j + 1);
                const double c = immediate<KIND>(M, S, A, dp.x, after);
                if (!SURVIVAL) acc += dp.y * c;                           // Recursion.java:139
                bool bankrupt;
                const int ni = successor32<KIND>(M, S, A, __double2loint(gi.y), c, after, bankrupt);
                double vn = __ldg(Vn + ni);
                if (SURVIVAL && bankrupt) vn = 0.0;                       // RiskRecursion.java:87-95
                acc += gi.x * vn;                                         // Recursion.java:142
            }
        } else {
            for (int j = 0; j < D; j++) {
                double after;
                const double2 dp = __ldg(rec + 2 * j), gi = __ldg(rec + 2 * j + 1);
                const double c = immediate<KIND>(M, S, A, dp.x, after);
                if (!SURVIVAL) acc += dp.y * c;                           // Recursion.java:139
                bool bankrupt;
                const long long ni = successor<KIND>(M, S, A, __double2loint(gi.y), c, after, bankrupt);
                double vn = __ldg(Vn + ni);
                if (SURVIVAL && bankrupt) vn = 0.0;                       // RiskRecursion.java:87-95
                acc += gi.x * vn;                                         // Recursion.java:142
            }
        }
        // ascending i within a lane: strict compare keeps the first optimum (Recursion.java:146-157)
        if (IS_MIN ? (acc < best) : (acc > best)) { best = acc; besti = i; }
    }

    if (G > 1) {
#pragma unroll
        for (int s = G / 2; s > 0; s >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, s, G);
            const int oi = __shfl_xor_sync(0xffffffffu, besti, s, G);
            if (better<IS_MIN>(ov, oi, best, besti)) { best = ov; besti = oi; }
        }
    }
    if (live && lane == 0) {
        Vt[idx] = best;
        Qt[idx] = besti == kNoAction ? -1 : besti;
    }
}

// Lead-time backorder models, one warp per state: everything that depends on the demand alone —
// (p_j, p_j*gamma), the holding+penalty term at level y - d_j and the successor's row offset — is
// tabulated per warp in shared memory once, so an evaluation is LDS + 5 fp64 instructions + the
// V_{t+1} gather (unit-stride across lanes: the successor's last pipeline slot is the action).
// Each lane carries 4 actions at a time for instruction-level parallelism.
// ((fv + hold) + pen) == fv + (hold + pen) bit for bit because one of hold/pen is always +0.
struct StagedRow { double L; long long row; };

template <bool IS_MIN, bool DEDUP>
__global__ void __launch_bounds__(256)
bi_backorder_staged(const __grid_constant__ DevModel M, const int t, const int D, const int pmf_off,
                    const double* __restrict__ Vn, double* __restrict__ Vt, int* __restrict__ Qt,
                    const long long lo, const long long hi) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* PP = reinterpret_cast<double2*>(smem_raw);                       // [D] (p, p*gamma)
    StagedRow* LR = reinterpret_cast<StagedRow*>(smem_raw + (size_t)D * 16);  // [8 warps][D]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Which 8 states share a CTA.  Lead time 1, and every folded (DEDUP) grid: 8 consecutive indices
    // already differ in the level y only, so their warps read the same successor rows one demand
    // step apart.  Lead time 2 on the real grid: consecutive indices differ in preQ2, i.e. in the
    // COLUMN block, and share nothing — so a CTA takes 8 consecutive preQ1 for one (x, preQ2) instead:
    // 8 warps x D demands then touch 8 + D - 1 rows instead of 8 * D and L1 serves the rest.
    long long idx;
    if (M.lead == 2 && !DEDUP) {
        const int groups = (M.nQ + 7) >> 3;                       // preQ1 groups of 8
        const long long first = lo / ((long long)M.nQ * M.nQ);    // first inventory row of the shard
        long long b = blockIdx.x;
        const int q2 = (int)(b % M.nQ); b /= M.nQ;
        const int g = (int)(b % groups); b /= groups;
        const int q1 = g * 8 + warp;
        idx = ((first + b) * M.nQ + q1) * M.nQ + q2;
        if (q1 >= M.nQ) idx = -1;
    } else {
        idx = lo + (long long)blockIdx.x * 8 + warp;
    }
    const bool live = idx >= lo && idx < hi;
    const StateCtx S = decode_state<SDPB_COST_BACKORDER>(M, t, live ? idx : lo, DEDUP);
    for (int j = threadIdx.x; j < D; j += 256)
        PP[j] = make_double2(M.pmf_p[pmf_off + j], M.pmf_pg[pmf_off + j]);
    StagedRow* my = LR + (size_t)warp * D;
    const double stock = S.x + S.q1;  // Leadtime.java:64,75
    const int iy = S.ix + S.iq1;
    for (int j = lane; j < D; j += 32) {
        const double lvl = stock - M.pmf_d[pmf_off + j];
        const double hold = M.h * fmax(lvl, 0.0);
        const double pen = M.pen * fmax(-lvl, 0.0);
        int il = iy - M.pmf_di[pmf_off + j];
        if (S.lost) il = max(il, M.i_zero);
        il = min(il, M.nI - 1);
        il = max(il, 0);
        my[j].L = hold + pen;
        my[j].row = il * S.strideX;
    }
    __syncthreads();

    double best = IS_MIN ? DBL_MAX : -DBL_MAX;
    int besti = kNoAction;
    const long long pipe_q2 = (M.lead == 2) ? (long long)S.iq2 * M.nQ : 0;
    for (int base = 0; base < S.nA; base += 128) {
        double fv[4], acc[4];
        long long pipe[4];
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int i = min(base + 32 * r + lane, S.nA - 1);  // out-of-range lanes recompute a valid action
            const double a = (double)i * M.step;
            fv[r] = (a > 0.0 ? M.K : 0.0) + S.v * a;
            pipe[r] = pipe_q2 + i;
            acc[r] = 0.0;
        }
        if (Vn == nullptr) {
            for (int j = 0; j < D; j++) {
                const double2 pp = PP[j];
                const double L = my[j].L;
#pragma unroll
                for (int r = 0; r < 4; r++) acc[r] += pp.x * (fv[r] + L);
            }
        } else {
#pragma unroll 2
            for (int j = 0; j < D; j++) {
                const double2 pp = PP[j];
                const StagedRow lr = my[j];
                const double* __restrict__ row = Vn + lr.row;
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const double vn = __ldg(row + pipe[r]);
                    acc[r] += pp.x * (fv[r] + lr.L);
                    acc[r] += pp.y * vn;
                }
            }
        }
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int i = base + 32 * r + lane;
            if (i < S.nA && (IS_MIN ? (acc[r] < best) : (acc[r] > best))) { best = acc[r]; besti = i; }
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, s);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, s);
        if (better<IS_MIN>(ov, oi, best, besti)) { best = ov; besti = oi; }
    }
    if (live && lane == 0) {
        Vt[idx] = best;
        Qt[idx] = besti == kNoAction ? -1 : besti;
    }
}

// Broadcast the virtual tables H(y, [preQ2], [cash]) to every real state (x, preQ, ...) of [lo, hi).
template <int KIND>
__global__ void __launch_bounds__(256)
expand_dedup(const __grid_constant__ DevModel M, const double* __restrict__ Hv, const int* __restrict__ Ha,
             double* __restrict__ Vt, int* __restrict__ Qt, const long long lo, const long long hi) {
    const long long idx = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= hi) return;
    long long r = idx;
    int iw = 0, iq2 = 0;
    if (KIND != SDPB_COST_BACKORDER) { iw = (int)(r % M.nW); r /= M.nW; }
    if (M.lead >= 2) { iq2 = (int)(r % M.nQ); r /= M.nQ; }
    const int iq1 = (int)(r % M.nQ);
    const long long iy = r / M.nQ + iq1;
    long long v = iy;
    if (M.lead >= 2) v = v * M.nQ + iq2;
    if (KIND != SDPB_COST_BACKORDER) v = v * M.nW + iw;
    Vt[idx] = Hv[v];
    Qt[idx] = Ha[v];
}

// One thread per (state of period t): if the state is reached, mark every successor in the
// period t+1 mask.  Masks are one byte per state; races only ever write 1.
template <int KIND, bool SURVIVAL>
__global__ void __launch_bounds__(256)
reach_forward(const __grid_constant__ DevModel M, const int t, const int D, const int pmf_off,
              const unsigned char* __restrict__ mask_t, unsigned char* __restrict__ mask_n,
              unsigned long long* __restrict__ counters) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M.S || !mask_t[idx]) return;
    const StateCtx S = decode_state<KIND>(M, t, idx);
    const double* __restrict__ pd = M.pmf_d + pmf_off;
    const int* __restrict__ pdi = M.pmf_di + pmf_off;
    // dense-grid artefacts at a state the reference visits: [0] clipped successors, [1] capped action sets,
    // [2] successors whose cash hit a bound (see successor_clip)
    unsigned n_clip = 0, n_cash = 0;
    const bool has_next = mask_n != nullptr;  // period T: the recursion stops (no transition is evaluated)
    for (int i = 0; has_next && i < S.nA; i++) {
        const ActionCtx A = prep_action<KIND>(M, S, i);
        for (int j = 0; j < D; j++) {
            double after;
            const double c = immediate<KIND>(M, S, A, __ldg(pd + j), after);
            bool bankrupt;
            const long long ni = successor<KIND>(M, S, A, __ldg(pdi + j), c, after, bankrupt);
            const unsigned clip = successor_clip<KIND>(M, S, A, __ldg(pdi + j), c, after);
            n_clip += clip & 1u;
            n_cash += (clip >> 1) & 1u;
            // getSurvProb never recurses into a bankrupt successor (RiskRecursion.java:89-94)
            if (!(SURVIVAL && bankrupt)) mask_n[ni] = 1;
        }
    }
    if (n_clip) atomicAdd(counters + 0, (unsigned long long)n_clip);
    if (S.capped) atomicAdd(counters + 1, 1ull);
    if (n_cash) atomicAdd(counters + 2, (unsigned long long)n_cash);
}

// One thread per sample path: roll the solved policy forward (Simulation.java:59-70).
template <int KIND>
__global__ void __launch_bounds__(128)
simulate_paths(const __grid_constant__ DevModel M, const long long init_idx, const double* __restrict__ samples,
               const int n, const double* __restrict__ disc_pow, const int* const* __restrict__ Qt,
               double* __restrict__ values, int* __restrict__ off_grid) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long idx = init_idx;
    double sum = 0.0;
    for (int t = 1; t <= M.T; t++) {
        const StateCtx S = decode_state<KIND>(M, t, idx);
        int qi = Qt[t - 1][idx];
        if (qi < 0) qi = 0;  // bestOrderQty stayed 0
        const ActionCtx A = prep_action<KIND>(M, S, qi);
        const double d = (double)jround(samples[(size_t)i * M.T + (t - 1)]);  // Math.round(samples[i][t])
        const double dq = d / M.step;
        if (dq != floor(dq)) atomicAdd(off_grid, 1);
        double after;
        const double c = immediate<KIND>(M, S, A, d, after);
        sum += disc_pow[t - 1] * c;
        bool bankrupt;
        idx = successor<KIND>(M, S, A, (int)dq, c, after, bankrupt);
    }
    values[i] = sum;
}

// One thread per (state, action, demand) triple: the lambdas alone, for descriptor spot checks.
template <int KIND>
__global__ void eval_triples(const __grid_constant__ DevModel M, const int t, const int n,
                             const long long* __restrict__ sidx, const int* __restrict__ aidx,
                             const double* __restrict__ dem, const int* __restrict__ demi,
                             double* __restrict__ c_out, long long* __restrict__ next_out,
                             int* __restrict__ na_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const StateCtx S = decode_state<KIND>(M, t, sidx[i]);
    const ActionCtx A = prep_action<KIND>(M, S, aidx[i]);
    double after;
    const double c = immediate<KIND>(M, S, A, dem[i], after);
    bool bankrupt;
    c_out[i] = c;
    next_out[i] = successor<KIND>(M, S, A, demi[i], c, after, bankrupt);
    na_out[i] = S.nA;
}

}  // namespace sdpb
