// reached.cu — the reference's two-product recursions on the GPU, over the states they REACH.
//
//   kind 0  src/sdp/cash/multiItem/CashRecursionMultiLead.java:54-95 (loop, `> val + 0.1` acceptance rule)
//           src/cash/overdraft/MultiProductLeadtime.java:150-224 (action list, immediate value, transition)
//   kind 1  src/sdp/cash/multiItem/CashRecursionMultiXR.java:61-95, lambdas src/cash/multiItem/MultiItemCashXR.java:73-126
//           (state (x1, x2, R), actions = order-up-to pairs, `(int)` casts)
//   kind 2  src/sdp/cash/multiItem/CashRecursionV.java:83-131 (V / Pi form: no immediate value, `> val + 0.01`,
//           V_{T+1} = boundFinalCash), lambdas src/cash/multiItem/MultiItemYR.java:89-146
//   kind 3  src/sdp/cash/CashRecursion.java:79-140 with the lambdas of src/cash/singleItem/CashConstraintTest.java:76-116
//           (one product; both state components rounded as Math.round(v * 0.1) / 0.1, so neither axis has an exact step)
//
// (what follows describes kind 0, for which the engine was written; the other two plug their lambdas into it)
//
// State (period, x1, x2, preQ1, preQ2, cash): the cash balance is NOT quantised (MultiProductLeadtime.java:219 is
// commented out), so the state space is not a grid and the dense kernels of sdpb200.cu do not apply -- this is the
// model the reference's author gave up on ("3 hour no solution", MultiProductLeadtime.java:28).  The reference
// memoises top-down; here the same set of states is built bottom-up:
//
//   forward   F_1 = {initial state};  F_{t+1} = unique{ f(s, a, d) : s in F_t, a in A, d in D_t }   (expand, sort, unique)
//   backward  V_T on F_T, then V_t on F_t with V_{t+1}(f(s,a,d)) found by binary search in the sorted F_{t+1}
//
// A solve is a handle (sdpb_reached_open) that keeps, per period, the sorted keys, V and the action index of the
// reached states, so that every reached state can be queried (ml_query), the handle extended with states of any period
// (ml_extend: only the states no earlier call reached are expanded -- N_t = (successors of N_{t-1} u roots of t) \ F_t,
// membership by binary search (ml_known) -- and solved against the merged F_{t+1}, then merged into F_t by key), and
// the policy rolled out over sample paths (ml_simulate), extending the handle with the states the paths meet.
// sdpb_reached_solve is open -> read the root -> destroy.
//
// The arithmetic of every (s, a, d) is the reference's, operation for operation and in its order (no FMA: the file is
// compiled with -fmad=false); the action scan is serial in the reference's i-major order because the acceptance rule
// `value > best + 0.1` is order dependent.  Two thread mappings: a thread per state (large frontiers: the last
// period of the T = 3 instance has 1.7e7 states x 2500 actions x 4 demand pairs) and a thread per (state, action)
// pair followed by a per-state scan (small frontiers, where a thread per state would leave the GPU empty).
#include <cuda_runtime.h>
#include <thrust/execution_policy.h>
#include <thrust/remove.h>
#include <thrust/sort.h>
#include <thrust/unique.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <exception>
#include <string>
#include <vector>

#include "../../include/sdpb200.h"
#include "memo_tables.cuh"

namespace {

struct MLState {
    int x1, x2, q1, q2;
    double cash;
};

// sort / search key: the four integers packed, then the cash as an order-preserving word, so that the keys sort in the
// reference's memo-map order (t, x1, x2, preQ1, preQ2, cash) with cash compared numerically (CashRecursionMultiLead.java:45-51).
// The all-ones key marks a slot of an unlisted action: it sorts last and no state has it (q_bound <= 65535 keeps
// preQ2 below 0xffff).
struct MLKey {
    unsigned long long a, b;
};
struct MLKeyLess {
    __host__ __device__ bool operator()(const MLKey& l, const MLKey& r) const { return l.a < r.a || (l.a == r.a && l.b < r.b); }
};
struct MLKeyEq {
    __host__ __device__ bool operator()(const MLKey& l, const MLKey& r) const { return l.a == r.a && l.b == r.b; }
};
struct MLFlagged {
    __host__ __device__ bool operator()(unsigned char f) const { return f != 0; }
};

// order-preserving encoding of a double: set the sign bit of a non-negative value, flip every bit of a negative one
// (branch-free for the reason at ml_dec; topdown.cu's td_enc keeps a select: see there)
__host__ __device__ inline unsigned long long ml_enc(double v) {
    v += 0.0;  // -0.0 and +0.0 are one key in the reference's map (compared with ==)
    unsigned long long b;
    memcpy(&b, &v, sizeof b);
    return b ^ ((unsigned long long)((long long)b >> 63) | 0x8000000000000000ull);  // branch-free: see ml_dec
}
__host__ __device__ inline double ml_dec(unsigned long long b) {
    // branch-free (a select here costs the backward kernels 18 registers and 6 % more fp64 instructions)
    b ^= (unsigned long long)((long long)~b >> 63) | 0x8000000000000000ull;
    double v;
    memcpy(&v, &b, sizeof v);
    return v;
}

struct MLParams {
    int kind;  // sdpb_reached_kind
    double dr; // depositeRate of the XR / YR lambdas, interestRate of CashConstraintTest
    double K, h, min_cash_req, sq;  // CASH_ROUNDED: fixed cost, holding cost, minCashRequired, rounding factor q
    int T, Q, Q2, nD;  // the action list has Q * Q2 entries (Q2 = Q for the two-product kinds, 1 for one product)
    double price1, price2, v1, v2, sal1, sal2;
    double r0, r1, r2, limit, interest_free;
    double min_inv, max_inv, min_cash, max_cash, gamma, tie;
    const double* d1;   // [T * nD] demand of product 1 (cast to int as the reference does)
    const double* d2;
    const double* p;    // [T * nD]
    const double* pg;   // p * gamma
    const double* ovh;  // [T]
    const int* nDt;     // [T] demand points of each period (<= nD, the row stride)
};

__host__ __device__ inline MLKey ml_key(const MLState& s) {
    MLKey k;
    k.a = ((unsigned long long)(unsigned)s.x1 << 48) | ((unsigned long long)(unsigned)s.x2 << 32) |
          ((unsigned long long)(unsigned)s.q1 << 16) | (unsigned long long)(unsigned)s.q2;
    k.b = ml_enc(s.cash);
    return k;
}

__host__ __device__ inline MLState ml_state(const MLKey& k) {
    MLState s;
    s.x1 = (int)((k.a >> 48) & 0xffff); s.x2 = (int)((k.a >> 32) & 0xffff);
    s.q1 = (int)((k.a >> 16) & 0xffff); s.q2 = (int)(k.a & 0xffff);
    s.cash = ml_dec(k.b);
    return s;
}

__device__ __forceinline__ double jmax0(double x) { return x > 0.0 ? x : 0.0; }  // Math.max(0, x) for non-NaN x
__device__ __forceinline__ double jmin(double a, double b) { return a < b ? a : b; }

// MultiProductLeadtime.java:162-198
__device__ __forceinline__ double ml_immediate(const MLParams& P, int t, bool last, const MLState& s, int a1, int a2, int d1,
                                               int d2) {
    const double action1 = (double)a1, action2 = (double)a2, demand1 = (double)d1, demand2 = (double)d2;
    const double stock1 = (double)s.x1 + (double)s.q1, stock2 = (double)s.x2 + (double)s.q2;
    const double endInventory1 = jmax0(stock1 - demand1);
    const double endInventory2 = jmax0(stock2 - demand2);
    const double revenue1 = P.price1 * jmin(demand1, stock1);
    const double revenue2 = P.price2 * jmin(stock2, demand2);
    const double revenue = revenue1 + revenue2;
    const double orderingCosts = P.v1 * action1 + P.v2 * action2;
    double salValue = 0.0;
    if (last) salValue = P.sal1 * endInventory1 + P.sal2 * endInventory2;
    const double before = (s.cash - orderingCosts) - P.ovh[t - 1];
    double interest;
    if (before >= 0.0) interest = -P.r0 * before;
    else if (before >= -P.interest_free) interest = 0.0;
    else if (before >= -P.limit) interest = P.r1 * (-before - P.interest_free);
    else interest = P.r2 * (-before - P.limit) + P.r1 * (P.limit - P.interest_free);
    const double after = ((before - interest) + revenue) + salValue;
    return after - s.cash;
}

// MultiProductLeadtime.java:202-224 (the asymmetric clamps are the reference's)
__device__ __forceinline__ MLState ml_transition(const MLParams& P, const MLState& s, int a1, int a2, int d1, int d2, double c) {
    double e1 = jmax0(((double)s.x1 + (double)s.q1) - (double)d1);
    double e2 = jmax0(((double)s.x2 + (double)s.q2) - (double)d2);
    double nextCash = s.cash + c;
    nextCash = nextCash > P.max_cash ? P.max_cash : nextCash;
    nextCash = nextCash < P.min_cash ? P.min_cash : nextCash;
    e1 = e1 > P.max_inv ? P.max_inv : e1;
    e2 = e2 < P.min_inv ? P.min_inv : e2;
    MLState n;
    n.x1 = (int)e1; n.x2 = (int)e2; n.q1 = a1; n.q2 = a2; n.cash = nextCash;
    return n;
}

__device__ __forceinline__ long long ml_find(const MLKey* __restrict__ F, long long n, const MLKey& k) {
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        const MLKey m = F[mid];
        if (m.a < k.a || (m.a == k.a && m.b < k.b)) lo = mid + 1; else hi = mid;
    }
    return lo;  // the key is present by construction
}

struct MLTraits {  // the key of the memo tables (memo_tables.cuh)
    typedef MLKey Key;
    typedef MLKeyLess Less;
    typedef MLKeyEq Eq;
    static __device__ __forceinline__ long long lower(const MLKey* __restrict__ F, long long n, const MLKey& k) {
        return ml_find(F, n, k);
    }
};

// ---- kind 1: MultiItemCashXR.java:87-126 ----
__device__ __forceinline__ double xr_immediate(const MLParams& P, bool last, const MLState& s, double action1, double action2,
                                               double demand1, double demand2) {
    const double endInventory1 = jmax0(action1 - demand1);
    const double endInventory2 = jmax0(action2 - demand2);
    const double revenue1 = P.price1 * (action1 - endInventory1);
    const double revenue2 = P.price2 * (action2 - endInventory2);
    const double revenue = revenue1 + revenue2;
    const double initialCash = (s.cash - P.v1 * (double)s.x1) - P.v2 * (double)s.x2;
    const double orderingCostsY = P.v1 * action1 + P.v2 * action2;
    double salValue = 0.0;
    if (last) salValue = P.sal1 * endInventory1 + P.sal2 * endInventory2;
    return ((revenue + (1.0 - P.dr) * (s.cash - orderingCostsY)) + salValue) - initialCash;
}

__device__ __forceinline__ MLState xr_transition(const MLParams& P, const MLState& s, double a1, double a2, double d1, double d2,
                                                 double c) {
    double e1 = jmax0(a1 - d1), e2 = jmax0(a2 - d2);
    const double initialCash = (s.cash - P.v1 * (double)s.x1) - P.v2 * (double)s.x2;
    double nextCash = initialCash + c;
    nextCash = nextCash > P.max_cash ? P.max_cash : nextCash;
    nextCash = nextCash < P.min_cash ? P.min_cash : nextCash;
    e1 = e1 > P.max_inv ? P.max_inv : e1;
    e2 = e2 < P.min_inv ? P.min_inv : e2;
    nextCash = (double)(int)nextCash;
    MLState n;
    n.x1 = (int)e1; n.x2 = (int)e2; n.q1 = 0; n.q2 = 0;
    n.cash = (nextCash + P.v1 * (double)n.x1) + P.v2 * (double)n.x2;  // nextR
    return n;
}

// ---- kind 2: MultiItemYR.java:122-146 (Math.round(x * 10) / 10 is a LONG division) ----
__device__ __forceinline__ long long ml_jround(double x) {
    return __double2ll_rd(__dadd_rd(x, 0.5));  // floor of the exact x + 1/2: see jround() in dev_model.cuh
}

__device__ __forceinline__ MLState yr_transition(const MLParams& P, double y1, double y2, double iniR, double d1, double d2) {
    double e1 = jmax0(y1 - d1), e2 = jmax0(y2 - d2);
    const double revenue1 = P.price1 * jmin(y1, d1);
    const double revenue2 = P.price2 * jmin(y2, d2);
    double nextW = (revenue1 + revenue2) + (1.0 + P.dr) * ((iniR - P.v1 * y1) - P.v2 * y2);
    e1 = (double)(ml_jround(e1 * 10.0) / 10);
    e2 = (double)(ml_jround(e2 * 10.0) / 10);
    nextW = (double)(ml_jround(nextW * 10.0) / 10);
    nextW = nextW > P.max_cash ? P.max_cash : nextW;
    nextW = nextW < P.min_cash ? P.min_cash : nextW;
    e1 = e1 > P.max_inv ? P.max_inv : e1;
    e2 = e2 < P.min_inv ? P.min_inv : e2;
    MLState n;
    n.x1 = (int)e1; n.x2 = (int)e2; n.q1 = 0; n.q2 = 0; n.cash = nextW;
    return n;
}

// ---- kind 3: CashConstraintTest.java:76-116 (one product; x = k / q with k kept in the key) ----
__device__ __forceinline__ double cct_immediate(const MLParams& P, bool last, double x, double w, double action, double d) {
    const double revenue = P.price1 * jmin(x + action, d);
    const double fixedCost = action > 0.0 ? P.K : 0.0;
    const double variableCost = P.v1 * action;
    const double inventoryLevel = (x + action) - d;
    const double holdCosts = P.h * jmax0(inventoryLevel);
    const double interests = P.dr * (w - action * P.v1);
    double cashIncrement = (((revenue - fixedCost) - variableCost) - holdCosts) + interests;
    const double salValue = last ? P.sal1 * jmax0(inventoryLevel) : 0.0;
    cashIncrement += salValue;
    return cashIncrement;
}

__device__ __forceinline__ MLState cct_transition(const MLParams& P, double x, double w, double action, double d, double c) {
    double nextInventory = jmax0((x + action) - d);
    double nextCash = w + c;
    nextCash = nextCash > P.max_cash ? P.max_cash : nextCash;
    nextCash = nextCash < P.min_cash ? P.min_cash : nextCash;
    nextInventory = nextInventory > P.max_inv ? P.max_inv : nextInventory;
    nextInventory = nextInventory < P.min_inv ? P.min_inv : nextInventory;
    MLState n;
    n.cash = (double)ml_jround(nextCash * P.sq) / P.sq;   // Math.round(nextCash * 0.1) / 0.1
    n.x1 = (int)ml_jround(nextInventory * P.sq);           // the inventory is kept as k; its value is k / q
    n.x2 = 0; n.q1 = 0; n.q2 = 0;
    return n;
}

// the action with flat index ai of state s: its two components as the lambdas see them, and whether the reference's
// action list contains it (kind 2: `v1 * i + v2 * j < iniR + 0.1`, MultiItemYR.java:104-108)
__device__ __forceinline__ bool ml_action(const MLParams& P, const MLState& s, int ai, double& a1, double& a2) {
    const int i = ai / P.Q2, j = ai - i * P.Q2;
    if (P.kind == 0) { a1 = (double)i; a2 = (double)j; return true; }
    if (P.kind == 3) {  // CashConstraintTest.java:76-80
        a1 = (double)i; a2 = 0.0;
        const double maxQ = (double)(int)fmin((double)(P.Q - 1), fmax(0.0, ((s.cash - P.min_cash_req) - P.K) / P.v1));
        return i < (int)maxQ + 1;
    }
    a1 = (double)(s.x1 + i); a2 = (double)(s.x2 + j);  // order-up-to levels from (int) x
    if (P.kind == 1) return true;
    const double iniR = (s.cash + P.v1 * (double)s.x1) + P.v2 * (double)s.x2;
    return P.v1 * a1 + P.v2 * a2 < iniR + 0.1;
}

__device__ __forceinline__ MLState ml_successor(const MLParams& P, int t, const MLState& s, double a1, double a2, int j,
                                                double* c_out) {
    const double d1 = P.d1[(t - 1) * P.nD + j], d2 = P.d2[(t - 1) * P.nD + j];
    if (P.kind == 0) {
        const double c = ml_immediate(P, t, false, s, (int)a1, (int)a2, (int)d1, (int)d2);
        if (c_out) *c_out = c;
        return ml_transition(P, s, (int)a1, (int)a2, (int)d1, (int)d2, c);
    }
    if (P.kind == 1) {
        const double c = xr_immediate(P, false, s, a1, a2, d1, d2);
        if (c_out) *c_out = c;
        return xr_transition(P, s, a1, a2, d1, d2, c);
    }
    if (P.kind == 3) {
        const double x = (double)s.x1 / P.sq;
        const double c = cct_immediate(P, false, x, s.cash, a1, d1);
        if (c_out) *c_out = c;
        return cct_transition(P, x, s.cash, a1, d1, c);
    }
    const double iniR = (s.cash + P.v1 * (double)s.x1) + P.v2 * (double)s.x2;
    return yr_transition(P, a1, a2, iniR, d1, d2);
}

// F_{t+1} candidates: one entry per (state, action, demand)
__global__ void ml_expand(MLParams P, int t, const MLKey* __restrict__ F, long long nF, MLKey* __restrict__ out) {
    const long long A = (long long)P.Q * P.Q2;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= nF * A) return;
    const long long si = gid / A;
    const int ai = (int)(gid - si * A);
    const MLState s = ml_state(F[si]);
    double a1, a2;
    const bool feasible = ml_action(P, s, ai, a1, a2);
    // an action the reference's list does not contain reaches nothing: its slots repeat the state's first successor
    // under a listed action... there may be none, so they are filled with an all-ones key that unique() folds into
    // one entry and the caller drops
    const int nDt = P.nDt[t - 1];
    for (int j = 0; j < P.nD; j++) {
        MLKey k;
        if (feasible && j < nDt) k = ml_key(ml_successor(P, t, s, a1, a2, j, nullptr));
        else { k.a = ~0ull; k.b = ~0ull; }
        out[gid * P.nD + j] = k;
    }
}

// Q(s, a): kinds 0, 1: sum_j [ p_j c + (p_j gamma) V_{t+1}(f) ] (CashRecursionMultiLead.java:74-80,
// CashRecursionMultiXR.java:78-85); kind 2: sum_j p_j V_{t+1}(f) with V_{T+1} = boundFinalCash (CashRecursionV.java:88-97,125-128)
__device__ __forceinline__ double ml_action_value(const MLParams& P, int t, bool last, const MLState& s, double a1, double a2,
                                                  const MLKey* __restrict__ Fn, const double* __restrict__ Vn, long long nFn) {
    double q = 0.0;
    const int nDt = P.nDt[t - 1];
    for (int j = 0; j < nDt; j++) {
        const double pj = P.p[(t - 1) * P.nD + j];
        if (P.kind == 2) {
            const MLState n = ml_successor(P, t, s, a1, a2, j, nullptr);
            const double vn = last ? (n.cash + P.sal1 * (double)n.x1) + P.sal2 * (double)n.x2   // MultiItemYR.java:116-119
                                   : Vn[ml_find(Fn, nFn, ml_key(n))];
            q += pj * vn;
            continue;
        }
        const double d1 = P.d1[(t - 1) * P.nD + j], d2 = P.d2[(t - 1) * P.nD + j];
        const double x3 = (double)s.x1 / P.sq;  // kind 3: the inventory value
        const double c = P.kind == 0 ? ml_immediate(P, t, last, s, (int)a1, (int)a2, (int)d1, (int)d2)
                       : P.kind == 1 ? xr_immediate(P, last, s, a1, a2, d1, d2)
                                     : cct_immediate(P, last, x3, s.cash, a1, d1);
        q += pj * c;
        if (!last) {
            const MLState n = P.kind == 0 ? ml_transition(P, s, (int)a1, (int)a2, (int)d1, (int)d2, c)
                            : P.kind == 1 ? xr_transition(P, s, a1, a2, d1, d2, c)
                                          : cct_transition(P, x3, s.cash, a1, d1, c);
            q += P.pg[(t - 1) * P.nD + j] * Vn[ml_find(Fn, nFn, ml_key(n))];
        }
    }
    return q;
}

// a thread per state, serial i-major action scan with the `> val + tie` rule (CashRecursionMultiLead.java:81-85)
__global__ void ml_backward_state(MLParams P, int t, const MLKey* __restrict__ F, long long nF, const MLKey* __restrict__ Fn,
                                  const double* __restrict__ Vn, long long nFn, double* __restrict__ V, int* __restrict__ Qa) {
    const long long si = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (si >= nF) return;
    const MLState s = ml_state(F[si]);
    const bool last = t == P.T;
    double val = -DBL_MAX;
    int best = 0;  // bestActions = new Actions(0, 0); kind 2: bestYs = (x1, x2) = offsets (0, 0) as well
    const int A = P.Q * P.Q2;
    for (int ai = 0; ai < A; ai++) {
        double a1, a2;
        if (!ml_action(P, s, ai, a1, a2)) continue;
        const double q = ml_action_value(P, t, last, s, a1, a2, Fn, Vn, nFn);
        if (q > val + P.tie) { val = q; best = ai; }
    }
    V[si] = val;
    Qa[si] = best;
}

// small frontiers: a thread per (state, action) pair ...
__global__ void ml_backward_pairs(MLParams P, int t, const MLKey* __restrict__ F, long long nF, const MLKey* __restrict__ Fn,
                                  const double* __restrict__ Vn, long long nFn, double* __restrict__ QV) {
    const long long A = (long long)P.Q * P.Q2;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= nF * A) return;
    const long long si = gid / A;
    const int ai = (int)(gid - si * A);
    const MLState s = ml_state(F[si]);
    double a1, a2;
    // an action that is not in the reference's list can never be accepted: NaN fails `q > val + tie`
    QV[gid] = ml_action(P, s, ai, a1, a2) ? ml_action_value(P, t, t == P.T, s, a1, a2, Fn, Vn, nFn) : __longlong_as_double(0x7ff8000000000000ll);
}

// ... then the serial scan per state
__global__ void ml_scan_pairs(MLParams P, const double* __restrict__ QV, long long nF, double* __restrict__ V, int* __restrict__ Qa) {
    const long long si = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (si >= nF) return;
    const long long A = (long long)P.Q * P.Q2;
    double val = -DBL_MAX;
    int best = 0;
    for (long long ai = 0; ai < A; ai++) {
        const double q = QV[si * A + ai];
        if (q > val + P.tie) { val = q; best = (int)ai; }
    }
    V[si] = val;
    Qa[si] = best;
}

// the action getAction reports for a state with action index qi and value v: order quantities (i, j) for kinds 0 and 3,
// order-up-to levels (x1 + i, x2 + j) for kinds 1 and 2; a state without any accepted action keeps the reference's
// default, {0, 0} for kind 1 (new double[]{0, 0}) and (x1, x2) for kind 2 (bestYs = the offsets (0, 0))
__host__ __device__ inline void ml_reported_action(int kind, int q2, const MLState& s, int qi, double v, double& a1,
                                                   double& a2) {
    const int ai = qi / q2, aj = qi % q2;
    if (kind == 0 || kind == 3) { a1 = ai; a2 = aj; return; }
    const bool none = v == -DBL_MAX;
    a1 = kind == 1 && none ? 0.0 : (double)(s.x1 + ai);
    a2 = kind == 1 && none ? 0.0 : (double)(s.x2 + aj);
}

// listed actions of each state summed into *total (kinds 2 and 3, whose lists depend on the state)
__global__ void ml_count_actions(MLParams P, const MLKey* __restrict__ F, long long n, unsigned long long* __restrict__ total) {
    const long long si = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (si >= n) return;
    const MLState s = ml_state(F[si]);
    unsigned long long c = 0;
    for (int ai = 0; ai < P.Q * P.Q2; ai++) {
        double a1, a2;
        if (ml_action(P, s, ai, a1, a2)) c++;
    }
    atomicAdd(total, c);
}

// the filter of an extension: flag[i] = 1 when candidate i is already in the sorted table F
__global__ void ml_known(const MLKey* __restrict__ F, long long n, const MLKey* __restrict__ c, long long m,
                         unsigned char* __restrict__ flag) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const long long at = ml_find(F, n, c[i]);
    flag[i] = at < n && MLKeyEq()(F[at], c[i]) ? 1 : 0;
}

// One period of the roll-out for memo::memo_simulate: (a1, a2) = getAction(state), d = Math.round(sample),
// c(state, a, d) (salvage when t == T), state = f(state, a, d, c).  Kind 2 has no immediate value: a path is worth
// boundFinalCash of the state after period T.
struct MLStep {
    MLParams P;
    __device__ __forceinline__ bool operator()(int t, MLKey& s, int qi, double v, const double* smp, double& c) const {
        const MLState st = ml_state(s);
        double a1, a2;
        ml_reported_action(P.kind, P.Q2, st, qi, v, a1, a2);
        const double d1 = (double)ml_jround(smp[0]), d2 = P.kind != 3 ? (double)ml_jround(smp[1]) : 0.0;  // kind 3: one demand
        const bool last = t == P.T;
        if (P.kind == 2) {
            const double iniR = (st.cash + P.v1 * (double)st.x1) + P.v2 * (double)st.x2;
            const MLState nx = yr_transition(P, a1, a2, iniR, d1, d2);
            c = last ? (nx.cash + P.sal1 * (double)nx.x1) + P.sal2 * (double)nx.x2 : 0.0;  // MultiItemYR.java:116-119
            if (!last) s = ml_key(nx);
            return last;
        }
        const double x3 = (double)st.x1 / P.sq;  // kind 3: the inventory value
        c = P.kind == 0 ? ml_immediate(P, t, last, st, (int)a1, (int)a2, (int)d1, (int)d2)
          : P.kind == 1 ? xr_immediate(P, last, st, a1, a2, d1, d2)
                        : cct_immediate(P, last, x3, st.cash, a1, d1);
        if (!last)
            s = ml_key(P.kind == 0 ? ml_transition(P, st, (int)a1, (int)a2, (int)d1, (int)d2, c)
                       : P.kind == 1 ? xr_transition(P, st, a1, a2, d1, d2, c)
                                     : cct_transition(P, x3, st.cash, a1, d1, c));
        return false;
    }
};

thread_local std::string g_ml_error;

int ml_fail(int rc, const std::string& msg) {
    g_ml_error = msg;
    return rc;
}

}  // namespace

struct sdpb_reached {
    sdpb_reached_model m;  // scalars only: the caller's pointers are not kept
    MLParams P{};
    int device = 0;
    int n_int = 4;  // API-order coordinates before the cash: 4 | 2 | 2 | 1
    long long A = 0;
    long long scratch_bytes = 0;
    std::vector<int> lens;      // demand points of each period
    std::vector<void*> owned;   // model tables
    memo::Tables<MLTraits> mt;  // sorted in memo-map order; Q: the flat action index
};

namespace {

// N_t: the sorted roots of period t and the successors of the n_src new states `src` of period t - 1, minus the states
// the handle already holds in period t; sorted and unique, into a right-sized *out.  All candidates are expanded at
// once: a period whose candidates, with the sort's scratch, would pass the budget fails with SDPB_ERR_NOMEM.
int ml_new_states(sdpb_reached* h, int t, const MLKey* src, long long n_src, const std::vector<MLKey>& roots, MLKey** out,
                  long long* n_out) {
    *out = nullptr;
    *n_out = 0;
    const long long nr = (long long)roots.size(), pairs = n_src * h->A, cand = pairs * h->P.nD + nr;
    if (cand == 0) return SDPB_OK;
    cudaStream_t st = h->mt.stream;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const double budget = h->scratch_bytes > 0 ? (double)h->scratch_bytes : (double)free_b;
    if ((double)cand * sizeof(MLKey) * 2.2 > budget)
        return ml_fail(SDPB_ERR_NOMEM, "period " + std::to_string(t) + " has " + std::to_string(cand) + " candidate states: more than " +
                                           (h->scratch_bytes > 0 ? "a scratch budget of " + std::to_string(h->scratch_bytes) + " bytes"
                                                                 : std::string("this GPU's memory")) + " holds");
    memo::DevBuf buf;
    if (!buf.alloc((size_t)cand * sizeof(MLKey))) return ml_fail(SDPB_ERR_NOMEM, "allocation of the candidate states failed");
    MLKey* c = (MLKey*)buf.p;
    if (pairs > 0) {
        ml_expand<<<(unsigned)((pairs + 127) / 128), 128, 0, st>>>(h->P, t - 1, src, n_src, c);
        if (cudaGetLastError() != cudaSuccess) return ml_fail(SDPB_ERR_CUDA, "ml_expand launch failed");
    }
    if (nr > 0 && cudaMemcpyAsync(c + pairs * h->P.nD, roots.data(), (size_t)nr * sizeof(MLKey), cudaMemcpyHostToDevice, st) != cudaSuccess)
        return ml_fail(SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
    long long m = 0;
    const MLKey* Fo = h->mt.F[t - 1];
    const long long no = h->mt.nF[t - 1];
    try {
        auto par = thrust::cuda::par.on(st);
        thrust::sort(par, c, c + cand, MLKeyLess());
        m = (long long)(thrust::unique(par, c, c + cand, MLKeyEq()) - c);
        if (m > 0) {  // the slots of actions the reference's list does not contain sort last, as one key
            MLKey tail;
            if (cudaMemcpyAsync(&tail, c + m - 1, sizeof tail, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess)
                return ml_fail(SDPB_ERR_CUDA, std::string("forward pass: ") + cudaGetErrorString(cudaGetLastError()));
            if (tail.a == ~0ull && tail.b == ~0ull) m--;
        }
        if (m > 0 && no > 0) {  // keep what period t does not hold yet
            memo::DevBuf flag;
            if (!flag.alloc((size_t)m)) return ml_fail(SDPB_ERR_NOMEM, "allocation of the filter flags failed");
            ml_known<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(Fo, no, c, m, (unsigned char*)flag.p);
            if (cudaGetLastError() != cudaSuccess) return ml_fail(SDPB_ERR_CUDA, "ml_known launch failed");
            m = (long long)(thrust::remove_if(par, c, c + m, (const unsigned char*)flag.p, MLFlagged()) - c);
            if (cudaStreamSynchronize(st) != cudaSuccess) return ml_fail(SDPB_ERR_CUDA, "forward pass: filter");
        }
    } catch (const std::exception& ex) {
        return ml_fail(SDPB_ERR_CUDA, std::string("sort / unique: ") + ex.what());
    }
    if (m == 0) return SDPB_OK;
    if (!memo::alloc(*out, m)) return ml_fail(SDPB_ERR_NOMEM, "allocation of the states of period " + std::to_string(t) + " failed");
    *n_out = m;
    if (cudaMemcpyAsync(*out, c, (size_t)m * sizeof(MLKey), cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
        return ml_fail(SDPB_ERR_CUDA, std::string("forward pass: ") + cudaGetErrorString(cudaGetLastError()));
    return SDPB_OK;
}

// sum over the n states F of period t of |listed actions| * D_t
int ml_evals(sdpb_reached* h, int t, const MLKey* F, long long n, double& evals) {
    const double D = h->lens[t - 1];
    if (h->m.kind == SDPB_REACHED_MULTILEAD || h->m.kind == SDPB_REACHED_MULTI_XR) {  // every pair is listed
        evals += (double)n * (double)h->A * D;
        return SDPB_OK;
    }
    memo::DevBuf tot;
    unsigned long long listed = 0;
    if (!tot.alloc(sizeof listed)) return ml_fail(SDPB_ERR_NOMEM, "allocation failed");
    if (cudaMemsetAsync(tot.p, 0, sizeof listed, h->mt.stream) != cudaSuccess) return ml_fail(SDPB_ERR_CUDA, "cudaMemsetAsync failed");
    ml_count_actions<<<(unsigned)((n + 127) / 128), 128, 0, h->mt.stream>>>(h->P, F, n, (unsigned long long*)tot.p);
    if (cudaGetLastError() != cudaSuccess ||
        cudaMemcpyAsync(&listed, tot.p, sizeof listed, cudaMemcpyDeviceToHost, h->mt.stream) != cudaSuccess ||
        cudaStreamSynchronize(h->mt.stream) != cudaSuccess)
        return ml_fail(SDPB_ERR_CUDA, std::string("counting the actions: ") + cudaGetErrorString(cudaGetLastError()));
    evals += (double)listed * D;
    return SDPB_OK;
}

// getExpectedValue on the states roots[t - 1] of every period t >= p (each sorted and unique; empty for t < p): the
// forward pass builds the states no earlier call reached, the backward pass solves only those against the merged
// tables of the next period, and the merged tables of every touched period replace the handle's at the end.
int ml_extend(sdpb_reached* h, int p, const std::vector<std::vector<MLKey>>& roots) {
    const int T = h->m.T;
    memo::Stage<MLTraits> sg(T);
    if (cudaEventRecord(h->mt.e0, h->mt.stream) != cudaSuccess) return ml_fail(SDPB_ERR_CUDA, "cudaEventRecord failed");
    double evals = 0;
    for (int t = p; t <= T; t++) {
        const int k = t - 1;
        int rc = ml_new_states(h, t, t > p ? sg.N[k - 1] : nullptr, t > p ? sg.nN[k - 1] : 0, roots[k], &sg.N[k], &sg.nN[k]);
        if (rc == SDPB_OK && sg.nN[k] > 0) rc = ml_evals(h, t, sg.N[k], sg.nN[k], evals);
        if (rc != SDPB_OK) return rc;
    }
    auto backward = [h](int t, const MLKey* F, long long n, const MLKey* Fn, const double* Vn, long long nFn, double* V,
                        int* Q) {
        const long long A = h->A;
        cudaStream_t st = h->mt.stream;
        if (n * A <= 200000000LL && n < 50000) {  // few states: spread their actions over the GPU
            memo::DevBuf qv;
            if (!qv.alloc((size_t)(n * A) * sizeof(double))) return ml_fail(SDPB_ERR_NOMEM, "allocation of the action-value scratch failed");
            ml_backward_pairs<<<(unsigned)((n * A + 127) / 128), 128, 0, st>>>(h->P, t, F, n, Fn, Vn, nFn, (double*)qv.p);
            ml_scan_pairs<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(h->P, (const double*)qv.p, n, V, Q);
            return 2;
        }
        ml_backward_state<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(h->P, t, F, n, Fn, Vn, nFn, V, Q);
        return 1;
    };
    return memo::commit(h->mt, sg, p, evals, 0.0, backward, g_ml_error);
}

// The key of one API-order state: false when it has no key (an inventory or pipeline quantity that is not an integer
// in [0, 65535], or for kind 3 not k / state_q with such a k).  Coordinates must be finite.
bool ml_encode(const sdpb_reached* h, const double* s, MLKey& key) {
    double k[4] = {0, 0, 0, 0};
    for (int c = 0; c < h->n_int; c++) {
        k[c] = s[c];
        if (h->m.kind == SDPB_REACHED_CASH_ROUNDED) {  // the inventory is kept as k = round(x * q); x must be k / q exactly
            k[c] = std::floor(s[c] * h->m.state_q + 0.5);
            if (k[c] / h->m.state_q != s[c]) return false;
        }
        if (!(k[c] >= 0 && k[c] <= 65535) || k[c] != (double)(int)k[c]) return false;
    }
    MLState st;
    st.x1 = (int)k[0]; st.x2 = (int)k[1]; st.q1 = (int)k[2]; st.q2 = (int)k[3];
    st.cash = s[h->n_int];
    key = ml_key(st);
    return true;
}

bool ml_finite(const double* s, size_t n) {
    for (size_t i = 0; i < n; i++)
        if (!std::isfinite(s[i])) return false;
    return true;
}

// n API-order roots -> their keys, sorted and unique: SDPB_ERR_ARG for a coordinate that is not finite,
// SDPB_ERR_OFFGRID for a state without a key
int ml_root_keys(const sdpb_reached* h, const double* states, int n, std::vector<MLKey>& out) {
    const int nd = h->n_int + 1;
    if (!ml_finite(states, (size_t)n * nd)) return ml_fail(SDPB_ERR_ARG, "a state coordinate is not finite");
    out.resize((size_t)n);
    for (int i = 0; i < n; i++)
        if (!ml_encode(h, states + (size_t)i * nd, out[i]))
            return ml_fail(SDPB_ERR_OFFGRID, h->m.kind == SDPB_REACHED_CASH_ROUNDED
                                                 ? "the inventory of a state is not of the form k / state_q, k in [0, 65535]"
                                                 : "inventories and pipeline quantities must be integers in [0, 65535]");
    memo::canonical<MLTraits>(out);
    return SDPB_OK;
}

}  // namespace

extern "C" {

const char* sdpb_reached_last_error(void) { return g_ml_error.c_str(); }

void sdpb_reached_destroy(sdpb_reached* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    for (void* p : h->owned) cudaFree(p);
    delete h;  // and its memo tables
}

int sdpb_reached_open(const sdpb_reached_model* m, int device, int64_t scratch_bytes, const double* init_states, int n,
                      sdpb_reached** out) {
    g_ml_error.clear();
    if (!m || !out || n < 0 || (n > 0 && !init_states) || m->struct_size != sizeof(sdpb_reached_model))
        return ml_fail(SDPB_ERR_ARG, "bad argument / struct_size");
    *out = nullptr;
    if (scratch_bytes < 0) return ml_fail(SDPB_ERR_ARG, "scratch_bytes < 0");
    if (m->kind < SDPB_REACHED_MULTILEAD || m->kind > SDPB_REACHED_CASH_ROUNDED) return ml_fail(SDPB_ERR_ARG, "bad kind");
    if (m->kind == SDPB_REACHED_CASH_ROUNDED && !(m->state_q > 0.0 && m->vari_cost[0] > 0.0)) return ml_fail(SDPB_ERR_ARG, "CASH_ROUNDED needs state_q > 0 and a positive unit cost");
    if (m->T < 1 || m->q_bound < 1 || m->q_bound > 65535 || m->n_demands < 1 || !m->d1 || !m->d2 || !m->p || !m->overhead_t)
        return ml_fail(SDPB_ERR_ARG, "T, q_bound, n_demands must be positive and the tables non-null");
    if (!(m->max_inv <= 65535.0)) return ml_fail(SDPB_ERR_ARG, "max_inv must fit 16 bits");
    const int T = m->T, nD = m->n_demands;
    std::vector<int> lens(T, nD);
    if (m->n_demands_t)
        for (int t = 0; t < T; t++) {
            if (m->n_demands_t[t] < 1 || m->n_demands_t[t] > nD) return ml_fail(SDPB_ERR_ARG, "n_demands_t out of range");
            lens[t] = m->n_demands_t[t];
        }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return ml_fail(SDPB_ERR_NO_DEVICE, "no CUDA device (libsdpb200 has no CPU path)"); }
    if (device < 0) cudaGetDevice(&device);
    if (device >= ndev || cudaSetDevice(device) != cudaSuccess) return ml_fail(SDPB_ERR_NO_DEVICE, "cannot select the CUDA device");

    sdpb_reached* h = new (std::nothrow) sdpb_reached();
    if (!h) return ml_fail(SDPB_ERR_NOMEM, "out of host memory");
    h->m = *m;
    h->device = device;
    h->scratch_bytes = scratch_bytes;
    h->lens = lens;
    h->n_int = m->kind == SDPB_REACHED_MULTILEAD ? 4 : (m->kind == SDPB_REACHED_CASH_ROUNDED ? 1 : 2);
    const int q2 = m->kind == SDPB_REACHED_CASH_ROUNDED ? 1 : m->q_bound;
    h->A = (long long)m->q_bound * q2;
    auto bail = [&](int rc, std::string msg) { sdpb_reached_destroy(h); return ml_fail(rc, msg); };
    if (h->mt.open(T, g_ml_error) != SDPB_OK) return bail(SDPB_ERR_CUDA, g_ml_error);
    std::vector<double> pg((size_t)T * nD);
    for (size_t i = 0; i < pg.size(); i++) pg[i] = m->p[i] * m->gamma;  // first product of p * gamma * V
    auto upload = [&](const void* src, size_t bytes) -> void* {
        void* p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        h->owned.push_back(p);
        if (cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, h->mt.stream) != cudaSuccess) return nullptr;
        return p;
    };
    MLParams& P = h->P;
    P.kind = m->kind; P.dr = m->deposit_rate;
    P.K = m->fixed_cost; P.h = m->hold_cost; P.min_cash_req = m->min_cash_required; P.sq = m->state_q > 0.0 ? m->state_q : 1.0;
    P.T = T; P.Q = m->q_bound; P.Q2 = q2; P.nD = nD;
    P.price1 = m->price[0]; P.price2 = m->price[1]; P.v1 = m->vari_cost[0]; P.v2 = m->vari_cost[1];
    P.sal1 = m->salvage[0]; P.sal2 = m->salvage[1];
    P.r0 = m->r0; P.r1 = m->r1; P.r2 = m->r2; P.limit = m->limit; P.interest_free = m->interest_free;
    P.min_inv = m->min_inv; P.max_inv = m->max_inv; P.min_cash = m->min_cash; P.max_cash = m->max_cash;
    P.gamma = m->gamma; P.tie = m->tie_tolerance;
    const size_t tab = (size_t)T * nD * sizeof(double);
    P.d1 = (const double*)upload(m->d1, tab); P.d2 = (const double*)upload(m->d2, tab); P.p = (const double*)upload(m->p, tab);
    P.pg = (const double*)upload(pg.data(), tab); P.ovh = (const double*)upload(m->overhead_t, (size_t)T * sizeof(double));
    P.nDt = (const int*)upload(lens.data(), (size_t)T * sizeof(int));
    if (!P.d1 || !P.d2 || !P.p || !P.pg || !P.ovh || !P.nDt) return bail(SDPB_ERR_NOMEM, "allocation of the model tables failed");
    if (cudaStreamSynchronize(h->mt.stream) != cudaSuccess) return bail(SDPB_ERR_CUDA, "uploading the model tables failed");  // (pg, lens are locals)

    std::vector<std::vector<MLKey>> roots((size_t)T);
    int rc = ml_root_keys(h, init_states, n, roots[0]);
    if (rc == SDPB_OK && n > 0) rc = ml_extend(h, 1, roots);
    if (rc != SDPB_OK) return bail(rc, g_ml_error);
    *out = h;
    return SDPB_OK;
}

int sdpb_reached_value(sdpb_reached* h, int period, const double* states, int n, double* v, double* a1, double* a2) {
    g_ml_error.clear();
    if (!h) return ml_fail(SDPB_ERR_ARG, "null handle");
    if (period < 1 || period > h->m.T || n < 0 || (n > 0 && !states)) return ml_fail(SDPB_ERR_ARG, "bad period or states");
    if (n == 0) return SDPB_OK;
    const int nd = h->n_int + 1;
    if (!ml_finite(states, (size_t)n * nd)) return ml_fail(SDPB_ERR_ARG, "a state coordinate is not finite");
    std::vector<MLKey> keys((size_t)n);
    for (int i = 0; i < n; i++)
        if (!ml_encode(h, states + (size_t)i * nd, keys[i]))
            return ml_fail(SDPB_ERR_UNSOLVED, "state " + std::to_string(i) + " was not reached in period " + std::to_string(period));
    cudaSetDevice(h->device);
    std::vector<double> vv;
    std::vector<int> qi;
    const int rc = memo::lookup(h->mt, period, keys, vv, qi, g_ml_error);
    if (rc != SDPB_OK) return rc;
    for (int i = 0; i < n; i++) {
        double b1, b2;
        ml_reported_action(h->m.kind, h->P.Q2, ml_state(keys[i]), qi[i], vv[i], b1, b2);
        if (v) v[i] = vv[i];
        if (a1) a1[i] = b1;
        if (a2) a2[i] = b2;
    }
    return SDPB_OK;
}

int sdpb_reached_extend(sdpb_reached* h, int period, const double* states, int n) {
    g_ml_error.clear();
    if (!h) return ml_fail(SDPB_ERR_ARG, "null handle");
    if (period < 1 || period > h->m.T || n < 0 || (n > 0 && !states)) return ml_fail(SDPB_ERR_ARG, "bad period or states");
    if (n == 0) return SDPB_OK;
    std::vector<std::vector<MLKey>> roots((size_t)h->m.T);
    const int rc = ml_root_keys(h, states, n, roots[period - 1]);
    if (rc != SDPB_OK) return rc;
    cudaSetDevice(h->device);
    return ml_extend(h, period, roots);
}

int sdpb_reached_opt_table(sdpb_reached* h, double* rows, size_t* nrows) {
    g_ml_error.clear();
    if (!h || !nrows) return ml_fail(SDPB_ERR_ARG, "null argument");
    cudaSetDevice(h->device);
    auto row = [h](int t, const MLKey& k, double v, int qi, double* row) {  // the device order is the memo-map order
        const MLState s = ml_state(k);
        int c = 0;
        row[c++] = t;
        if (h->m.kind == SDPB_REACHED_CASH_ROUNDED) {
            row[c++] = (double)s.x1 / h->P.sq;
        } else {
            row[c++] = s.x1;
            row[c++] = s.x2;
            if (h->m.kind == SDPB_REACHED_MULTILEAD) { row[c++] = s.q1; row[c++] = s.q2; }
        }
        row[c++] = s.cash;
        ml_reported_action(h->m.kind, h->P.Q2, s, qi, v, row[c], row[c + 1]);
    };
    return memo::opt_table(h->mt, rows, nrows, h->n_int + 4, row, g_ml_error);
}

int sdpb_reached_states(const sdpb_reached* h, int64_t* n_states) {
    g_ml_error.clear();
    if (!h || !n_states) return ml_fail(SDPB_ERR_ARG, "null argument");
    for (int t = 0; t < h->m.T; t++) n_states[t] = h->mt.nF[t];
    return SDPB_OK;
}

int sdpb_reached_stats(const sdpb_reached* h, sdpb_stats* s) {
    g_ml_error.clear();
    if (!h || !s) return ml_fail(SDPB_ERR_ARG, "null argument");
    *s = h->mt.stats;
    return SDPB_OK;
}

int sdpb_reached_simulate(sdpb_reached* h, const double* init_state, const double* samples, int n, double discount,
                          double* values) {
    g_ml_error.clear();
    if (!h) return ml_fail(SDPB_ERR_ARG, "null handle");
    if (!init_state || !samples || !values || n < 1) return ml_fail(SDPB_ERR_ARG, "null argument or n < 1");
    if (h->m.kind == SDPB_REACHED_MULTI_YR && discount != 1.0)
        return ml_fail(SDPB_ERR_ARG, "the V / Pi form values a path by boundFinalCash alone: discount must be 1");
    if (!std::isfinite(discount)) return ml_fail(SDPB_ERR_ARG, "discount is not finite");
    const int T = h->m.T, nd = h->m.kind == SDPB_REACHED_CASH_ROUNDED ? 1 : 2;
    const size_t N = (size_t)n;
    if (!ml_finite(samples, N * T * nd)) return ml_fail(SDPB_ERR_ARG, "a sample is not finite");
    std::vector<std::vector<MLKey>> roots((size_t)T);
    int rc = ml_root_keys(h, init_state, 1, roots[0]);
    if (rc != SDPB_OK) return rc;
    cudaSetDevice(h->device);
    auto extend = [h](int p, const std::vector<std::vector<MLKey>>& r) { return ml_extend(h, p, r); };
    return memo::rollout(h->mt, MLStep{h->P}, roots[0][0], samples, n, nd, discount, extend, values, g_ml_error);
}

int sdpb_reached_solve(const sdpb_reached_model* m, int device, const double* init_state, double* value, double* action1,
                       double* action2, int64_t* n_states, double* solve_ms) {
    if (!init_state) return ml_fail(SDPB_ERR_ARG, "bad argument / struct_size");
    sdpb_reached* h = nullptr;
    int rc = sdpb_reached_open(m, device, 0, init_state, 1, &h);
    if (rc != SDPB_OK) return rc;
    rc = sdpb_reached_value(h, 1, init_state, 1, value, action1, action2);
    if (rc == SDPB_OK && n_states) sdpb_reached_states(h, n_states);
    if (rc == SDPB_OK && solve_ms) *solve_ms = h->mt.stats.solve_ms;
    sdpb_reached_destroy(h);
    return rc;
}

}  // extern "C"
