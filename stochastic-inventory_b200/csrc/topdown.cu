// topdown.cu — any single-product sdpb_model solved over the states its top-down recursion reaches.
//
// The reference answers getExpectedValue(state) for any real-valued state: it recurses top-down and memoises what it
// visits (Recursion.java:89-163).  The dense engine of sdpb200.cu needs every level, action and demand on a grid with a
// power-of-two step; this engine needs no grid.  It builds the reference's visit set period by period and solves it
// backwards on the device:
//
//   forward   F_1 = unique(initial states);  F_{t+1} = unique{ f(s, a, d) : s in F_t, a in A_t(s), d in D_t }  (t < T;
//             the survival recursion does not visit a successor with w' < 0, RiskRecursion.java:87-95)
//   backward  V_T on F_T, then V_t on F_t, V_{t+1}(f(s, a, d)) found by searching the sorted F_{t+1}
//
// A state is the key (x, preQ1, preQ2, w); two states are one key iff their coordinates are == as doubles (-0.0 is
// stored as +0.0).  Each coordinate is stored as an order-preserving 64-bit integer, the active coordinates packed
// first, so that a radix sort orders the keys as the reference's memo map does (t, x, q1, q2, w).
//
// A solved handle grows: getExpectedValue on states of any period (td_extend) expands only the states no earlier call
// reached, N_t = (successors of N_{t-1} u roots of t) \ F_t, solves them against the merged F_{t+1}, and merges
// (N_t, V, Q) into (F_t, V_t, Q_t) by key; V depends on the state alone, so nothing held changes.  A fresh solve is
// the extension of an empty handle with period-1 roots.  The policy roll-out (td_simulate) runs on the same tables and
// extends them with the states its paths meet, as the reference's getExpectedValue at every step does.
//
// The candidates of one period can be far more than memory holds (a cash model with ~1e6 states per period, 201
// actions and 200 demand points has 4e10), so the (state, feasible action) pairs are expanded in chunks bounded by the
// scratch budget; each chunk is compacted, sorted and uniqued, then merged into the running frontier.
//
// The arithmetic is the dense engine's generic kernel's (prep_action, immediate of kernel_generic.cuh), which restates
// the reference's lambdas operation for operation; the transition below follows the same lambdas on real values and
// clamps only where the flags or the lambdas clamp.  Compiled with -fmad=false like the rest.
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <thrust/execution_policy.h>
#include <thrust/merge.h>
#include <thrust/remove.h>
#include <thrust/scan.h>
#include <thrust/set_operations.h>
#include <thrust/unique.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <exception>
#include <string>
#include <vector>

#include "../../include/sdpb200.h"
#include "kernel_generic.cuh"
#include "memo_tables.cuh"

namespace {
using namespace sdpb;
typedef unsigned long long u64;

struct __align__(16) TDKey {
    u64 w[4];  // encoded (x, [q1], [q2], [w]): the active coordinates first, the rest 0
};
struct TDLess {
    __host__ __device__ bool operator()(const TDKey& a, const TDKey& b) const {
        for (int k = 0; k < 4; k++)
            if (a.w[k] != b.w[k]) return a.w[k] < b.w[k];
        return false;
    }
};
struct TDEq {
    __host__ __device__ bool operator()(const TDKey& a, const TDKey& b) const {
        return a.w[0] == b.w[0] && a.w[1] == b.w[1] && a.w[2] == b.w[2] && a.w[3] == b.w[3];
    }
};
// a filtered candidate slot: all ones, which no state encodes to (it would be a NaN inventory)
struct TDIsHole {
    __host__ __device__ bool operator()(const TDKey& k) const { return k.w[0] == ~0ull; }
};
// the radix sort sees only the ND active words, most significant first
template <int ND> struct TDDecomp;
template <> struct TDDecomp<1> {
    __host__ __device__ ::cuda::std::tuple<u64&> operator()(TDKey& k) const { return {k.w[0]}; }
};
template <> struct TDDecomp<2> {
    __host__ __device__ ::cuda::std::tuple<u64&, u64&> operator()(TDKey& k) const { return {k.w[0], k.w[1]}; }
};
template <> struct TDDecomp<3> {
    __host__ __device__ ::cuda::std::tuple<u64&, u64&, u64&> operator()(TDKey& k) const { return {k.w[0], k.w[1], k.w[2]}; }
};
template <> struct TDDecomp<4> {
    __host__ __device__ ::cuda::std::tuple<u64&, u64&, u64&, u64&> operator()(TDKey& k) const {
        return {k.w[0], k.w[1], k.w[2], k.w[3]};
    }
};

// order-preserving encoding of a double: set the sign bit of a non-negative value, flip every bit of a negative one
// (a select: reached.cu's branch-free ml_enc, the same mapping, changes every td_* kernel here and was not timed)
__host__ __device__ inline u64 td_enc(double v) {
    v += 0.0;  // -0.0 and +0.0 are one key (the memo map compares with ==)
    u64 b;
    memcpy(&b, &v, sizeof b);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double td_dec(u64 b) {
    b = (b >> 63) ? (b & 0x7fffffffffffffffull) : ~b;
    double v;
    memcpy(&v, &b, sizeof v);
    return v;
}

// the device model plus what only this engine needs
struct TDModel {
    DevModel M;
    double inv_max;  // the upper inventory clamp (the dense engine keeps it as the grid's last row)
    int lead;        // state shape: (x, [q1, [q2]], [w])
    int cash;
    __host__ __device__ int nd() const { return 1 + lead + cash; }
};

__host__ __device__ inline TDKey td_pack(const TDModel& P, double x, double q1, double q2, double w) {
    TDKey k;
    k.w[1] = k.w[2] = k.w[3] = 0;
    int n = 0;
    k.w[n++] = td_enc(x);
    if (P.lead >= 1) k.w[n++] = td_enc(q1);
    if (P.lead >= 2) k.w[n++] = td_enc(q2);
    if (P.cash) k.w[n++] = td_enc(w);
    return k;
}
__host__ __device__ inline void td_unpack(const TDModel& P, const TDKey& k, double& x, double& q1, double& q2, double& w) {
    int n = 0;
    x = td_dec(k.w[n++]);
    q1 = P.lead >= 1 ? td_dec(k.w[n++]) : 0.0;
    q2 = P.lead >= 2 ? td_dec(k.w[n++]) : 0.0;
    w = P.cash ? td_dec(k.w[n++]) : 0.0;
}

// what decode_state gives a grid point, for a real-valued state (grid indices stay 0: nothing here reads them)
template <int KIND>
__device__ __forceinline__ StateCtx td_state(const TDModel& P, int t, const TDKey& k, double& q2) {
    const DevModel& M = P.M;
    StateCtx S;
    S.t = t;
    S.ix = S.iq1 = S.iq2 = S.iw = 0;
    td_unpack(P, k, S.x, S.q1, q2, S.w);
    S.last = (t == M.T);
    S.price = M.price_t[t - 1];
    S.v = M.v_t[t - 1];
    S.ovh = M.ovh_t[t - 1];
    S.lost = (M.flags & SDPB_F_LOST_SALES) != 0;
    S.gy = (KIND == SDPB_COST_BACKORDER) && (M.flags & SDPB_F_GY_MODE) && t == 1;
    S.strideX = 0;
    feasible_actions<KIND>(M, S);
    return S;
}

// the cash quantiser on a real value; `t` is the period being left (TestPaper.java:107 rounds from q_from_period on)
__device__ __forceinline__ double td_quantise(const DevModel& M, double w, int t) {
    if (M.quantiser == SDPB_Q_TRUNC) {
        if (M.q_from_period > 0 && t >= M.q_from_period) w = (double)jround(w * M.q_mul) / M.q_div;
        return (double)(int)w;
    }
    const long long kk = jround(w * M.q_mul);
    if (M.quantiser == SDPB_Q_DIV) return (double)kk / M.q_div;
    return (double)(kk / M.q_idiv);  // Java long division
}

// f(s, a, d) on real values: CLSPTesting.java:89-94, Leadtime.java:61-68, CLSPforDraw.java:147-153 (backorder),
// CashConstraint.java:123-133, CashOverdraft.java:107-118, SingleProductLeadtime.java:106-119, cashSurvival.java:132-147,
// CashOverdraftTesting.java:103-111 (cash), CashConstraintXR.java:95-110 (XR: the successor's w is R = w' + v x').
// `bankrupt`: the successor's cash is negative (the survival recursion does not visit it).
template <int KIND>
__device__ __forceinline__ TDKey td_next(const TDModel& P, const StateCtx& S, double q2, const ActionCtx& A, double d,
                                         double c, double after, bool& bankrupt) {
    const DevModel& M = P.M;
    if (KIND == SDPB_COST_CASH_XR) {
        double nx = jmax0(A.stock - d);
        double nc = A.initCash + c;
        nc = nc > M.cash_max ? M.cash_max : nc;
        nc = nc < M.cash_min ? M.cash_min : nc;
        nx = nx > P.inv_max ? P.inv_max : nx;
        nx = nx < M.inv_min ? M.inv_min : nx;
        nc = td_quantise(M, nc, 1 << 30);  // the XR lambda quantises whatever the period
        const double nR = nc + S.v * nx;
        bankrupt = nR < 0.0;
        return td_pack(P, nx, 0.0, 0.0, nR);
    }
    double nx = A.stock - d, nw = 0.0;
    if (S.lost) nx = jmax0(nx);
    if (KIND != SDPB_COST_BACKORDER) {
        nw = (KIND == SDPB_COST_CASH_OD_TESTING) ? after : S.w + c;
        nw = nw > M.cash_max ? M.cash_max : nw;
        nw = nw < M.cash_min ? M.cash_min : nw;
    }
    if (M.flags & SDPB_F_CLAMP_INV) {  // upper clamp first (CLSPTesting.java:91-92)
        nx = nx > P.inv_max ? P.inv_max : nx;
        nx = nx < M.inv_min ? M.inv_min : nx;
    }
    if (KIND != SDPB_COST_BACKORDER) nw = td_quantise(M, nw, S.t);
    bankrupt = nw < 0.0;
    double nq1 = 0.0, nq2 = 0.0;
    if (M.lead == 1) nq1 = A.a;
    if (M.lead == 2) { nq1 = q2; nq2 = A.a; }
    return td_pack(P, nx, nq1, nq2, nw);
}

__device__ __forceinline__ bool td_less(const TDKey* __restrict__ F, long long i, const TDKey& k) {
    const ulonglong2 a = __ldg(reinterpret_cast<const ulonglong2*>(F + i));
    if (a.x != k.w[0]) return a.x < k.w[0];
    if (a.y != k.w[1]) return a.y < k.w[1];
    const ulonglong2 b = __ldg(reinterpret_cast<const ulonglong2*>(F + i) + 1);
    if (b.x != k.w[2]) return b.x < k.w[2];
    return b.y < k.w[3];
}

// first index of [lo, hi) whose key is not less than k
__device__ __forceinline__ long long td_lower(const TDKey* __restrict__ F, long long lo, long long hi, const TDKey& k) {
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (td_less(F, mid, k)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// The index of k in F[0, n) (present by construction), galloping from the previous demand's hit h.  The successors of
// one (s, a) over ascending d have non-increasing x', so consecutive hits are near each other: one row apart for the
// backorder models, about one inventory level's worth of cash states apart for the cash models.  Measured on one B200
// (1000 W): td_backward with this lookup runs 2.2e10 evaluations/s on C4 from (0, 0, 0) (3.1e11 in 14.4 s) and on C3
// from (0, 100) (1.1e11 in 4.7 s), a tenth of the solve; a plain binary search was not timed against it.
__device__ __forceinline__ long long td_find(const TDKey* __restrict__ F, long long n, const TDKey& k, long long h) {
    if (h < 0) return td_lower(F, 0, n, k);
    if (td_less(F, h, k)) {
        long long b = h, step = 1;
        while (b + step < n && td_less(F, b + step, k)) { b += step; step <<= 1; }
        return td_lower(F, b + 1, min(b + step, n), k);
    }
    long long b = h, step = 1;
    while (b - step >= 0 && !td_less(F, b - step, k)) { b -= step; step <<= 1; }
    return td_lower(F, max(b - step + 1, 0ll), b, k);
}

struct TDTraits {  // the key of the memo tables (memo_tables.cuh)
    typedef TDKey Key;
    typedef TDLess Less;
    typedef TDEq Eq;
    static __device__ __forceinline__ long long lower(const TDKey* __restrict__ F, long long n, const TDKey& k) {
        return td_lower(F, 0, n, k);
    }
};

// |A_t(s)| of every state; XR states whose order-up-to range was cut at max_order_idx + 1 are counted
template <int KIND>
__global__ void __launch_bounds__(256) td_count_actions(const __grid_constant__ TDModel P, const int t,
                                                        const TDKey* __restrict__ F, const long long n,
                                                        long long* __restrict__ nA, unsigned long long* __restrict__ capped) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double q2;
    const StateCtx S = td_state<KIND>(P, t, F[i], q2);
    nA[i] = S.nA;
    if (S.capped) atomicAdd(capped, 1ull);
}

// One thread per (state, feasible action) pair p of [p0, p0 + np): its D successors into out[j * np + (p - p0)], so
// that a warp's stores of one demand are contiguous (the order does not matter: the chunk is sorted next).  A
// successor equal to the previous demand's (clamped and lost-sales levels repeat) and, in the survival recursion, a
// bankrupt one are written as holes.  `off` = exclusive prefix sum of |A_t(s)| (n + 1 entries).
template <int KIND, bool SURVIVAL>
__global__ void __launch_bounds__(256) td_expand(const __grid_constant__ TDModel P, const int t, const int D,
                                                 const int pmf_off, const TDKey* __restrict__ F, const long long n,
                                                 const long long* __restrict__ off, const long long p0, const long long np,
                                                 TDKey* __restrict__ out) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= np) return;
    const long long p = p0 + g;
    long long lo = 0, hi = n;  // the state: last si with off[si] <= p
    while (hi - lo > 1) {
        const long long mid = (lo + hi) >> 1;
        if (off[mid] <= p) lo = mid; else hi = mid;
    }
    double q2;
    const StateCtx S = td_state<KIND>(P, t, F[lo], q2);
    const ActionCtx A = prep_action<KIND>(P.M, S, (int)(p - off[lo]));
    TDKey prev, hole;
    for (int k = 0; k < 4; k++) prev.w[k] = hole.w[k] = ~0ull;
    for (int j = 0; j < D; j++) {
        double after;
        const double d = P.M.pmf_d[pmf_off + j];
        const double c = immediate<KIND>(P.M, S, A, d, after);
        bool bankrupt;
        const TDKey k = td_next<KIND>(P, S, q2, A, d, c, after, bankrupt);
        const bool emit = !(SURVIVAL && bankrupt) && !TDEq()(k, prev);
        out[j * np + g] = emit ? k : hole;
        if (emit) prev = k;
    }
}

// V_t, Q_t on F_t: a warp per state, lanes over the actions (ascending within a lane, strict compare), then the
// lexicographic (value, action) shuffle reduction -- the first optimum in the reference's scan order wins.  The loop
// over the demands is the reference's (Recursion.java:129-161, RiskRecursion.java:66-104).
template <int KIND, bool SURVIVAL, bool IS_MIN>
__global__ void __launch_bounds__(256) td_backward(const __grid_constant__ TDModel P, const int t, const int D,
                                                   const int pmf_off, const TDKey* __restrict__ F, const long long n,
                                                   const TDKey* __restrict__ Fn, const double* __restrict__ Vn,
                                                   const long long nn, double* __restrict__ Vt, int* __restrict__ Qt) {
    const DevModel& M = P.M;
    const long long si = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const bool live = si < n;  // dead warps still take part in the shuffles
    double q2;
    const StateCtx S = td_state<KIND>(P, t, F[live ? si : 0], q2);
    double best = IS_MIN ? DBL_MAX : -DBL_MAX;
    int besti = kNoAction;
    const double* __restrict__ pd = M.pmf_d + pmf_off;
    const double* __restrict__ pp = M.pmf_p + pmf_off;
    const double* __restrict__ ppg = M.pmf_pg + pmf_off;
    for (int i = lane; live && i < S.nA; i += 32) {
        const ActionCtx A = prep_action<KIND>(M, S, i);
        double acc = 0.0;
        long long hit = -1;
        for (int j = 0; j < D; j++) {
            double after;
            const double d = __ldg(pd + j), p = __ldg(pp + j);
            const double c = immediate<KIND>(M, S, A, d, after);
            if (S.last) {
                if (!SURVIVAL) acc += p * c;                                 // Recursion.java:139
                else acc += p * ((S.w + c) >= 0.0 ? 1.0 : 0.0);              // RiskRecursion.java:80-84
                continue;
            }
            if (!SURVIVAL) acc += p * c;
            bool bankrupt;
            const TDKey k = td_next<KIND>(P, S, q2, A, d, c, after, bankrupt);
            double vn = 0.0;                                                 // RiskRecursion.java:87-95
            if (!(SURVIVAL && bankrupt)) {
                hit = td_find(Fn, nn, k, hit);
                vn = __ldg(Vn + hit);
            }
            acc += __ldg(ppg + j) * vn;                                      // Recursion.java:142
        }
        if (IS_MIN ? (acc < best) : (acc > best)) { best = acc; besti = i; }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, s);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, s);
        if (better<IS_MIN>(ov, oi, best, besti)) { best = ov; besti = oi; }
    }
    if (live && lane == 0) {
        Vt[si] = best;
        Qt[si] = besti == kNoAction ? -1 : besti;
    }
}

// One period of Simulation.java:59-70 for memo::memo_simulate: Q = getAction(state), d = Math.round(sample),
// c = the immediate value, state = f(s, Q, d).  f is applied whatever the cash: a survival model's roll-out goes on after
// a bankrupt period, as the reference's does.
template <int KIND>
struct TDStep {
    TDModel P;
    __device__ __forceinline__ bool operator()(int t, TDKey& s, int qi, double, const double* smp, double& c) const {
        if (qi < 0) qi = 0;  // bestOrderQty stayed 0
        double q2;
        const StateCtx S = td_state<KIND>(P, t, s, q2);
        const ActionCtx A = prep_action<KIND>(P.M, S, qi);
        const double d = (double)jround(*smp);  // Math.round(samples[i][t])
        double after;
        c = immediate<KIND>(P.M, S, A, d, after);
        bool bankrupt;
        if (t < P.M.T) s = td_next<KIND>(P, S, q2, A, d, c, after, bankrupt);
        return false;
    }
};

bool has_cash(const sdpb_model& m) { return m.cost_kind != SDPB_COST_BACKORDER; }

thread_local std::string g_td_error;

}  // namespace

struct sdpb_topdown {
    sdpb_model m;  // scalars only: the caller's pointers are not kept
    TDModel P{};
    int device = 0;
    int ndim = 1;
    unsigned allow = 0;
    long long scratch_bytes = 0;
    std::vector<int> pmf_len, pmf_off;
    std::vector<void*> owned;   // model tables
    memo::Tables<TDTraits> mt;  // action index -1: none improved on the initial value
    std::string err;
};

namespace {

int td_fail(sdpb_topdown* h, int rc, const std::string& msg) {
    if (h) h->err = msg; else g_td_error = msg;
    return rc;
}

template <int ND>
cudaError_t td_sort(void* tmp, size_t& tmp_bytes, cub::DoubleBuffer<TDKey>& keys, long long n, cudaStream_t s) {
    return cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, keys, n, TDDecomp<ND>(), s);
}
cudaError_t td_sort_nd(int nd, void* tmp, size_t& tmp_bytes, cub::DoubleBuffer<TDKey>& keys, long long n, cudaStream_t s) {
    switch (nd) {
    case 1: return td_sort<1>(tmp, tmp_bytes, keys, n, s);
    case 2: return td_sort<2>(tmp, tmp_bytes, keys, n, s);
    case 3: return td_sort<3>(tmp, tmp_bytes, keys, n, s);
    default: return td_sort<4>(tmp, tmp_bytes, keys, n, s);
    }
}

template <int KIND>
void launch_count(const sdpb_topdown* h, int t, const TDKey* F, long long n, long long* nA, unsigned long long* capped) {
    if (n == 0) return;
    td_count_actions<KIND><<<(unsigned)((n + 255) / 256), 256, 0, h->mt.stream>>>(h->P, t, F, n, nA, capped);
}
template <int KIND>
void launch_expand(const sdpb_topdown* h, int t, const TDKey* F, long long n, const long long* off, long long p0,
                   long long np, TDKey* out) {
    const int D = h->pmf_len[t - 1], po = h->pmf_off[t - 1];
    const unsigned blocks = (unsigned)((np + 255) / 256);
    if (h->m.recursion == SDPB_REC_SURVIVAL)
        td_expand<KIND, true><<<blocks, 256, 0, h->mt.stream>>>(h->P, t, D, po, F, n, off, p0, np, out);
    else
        td_expand<KIND, false><<<blocks, 256, 0, h->mt.stream>>>(h->P, t, D, po, F, n, off, p0, np, out);
}
// V, Q of the n states F of period t, against the sorted (Fn, Vn) of period t + 1 (nn states; none when t == T)
template <int KIND>
void launch_backward(const sdpb_topdown* h, int t, const TDKey* F, long long n, const TDKey* Fn, const double* Vn,
                     long long nn, double* V, int* Q) {
    const int D = h->pmf_len[t - 1], po = h->pmf_off[t - 1];
    if (n == 0) return;
    const unsigned blocks = (unsigned)((n + 7) / 8);
    if (h->m.recursion == SDPB_REC_SURVIVAL) {
        if constexpr (KIND == SDPB_COST_CASH_DEPOSIT || KIND == SDPB_COST_CASH_OVERDRAFT)
            td_backward<KIND, true, false><<<blocks, 256, 0, h->mt.stream>>>(h->P, t, D, po, F, n, Fn, Vn, nn, V, Q);
    } else if (h->m.direction == SDPB_MIN) {
        td_backward<KIND, false, true><<<blocks, 256, 0, h->mt.stream>>>(h->P, t, D, po, F, n, Fn, Vn, nn, V, Q);
    } else {
        td_backward<KIND, false, false><<<blocks, 256, 0, h->mt.stream>>>(h->P, t, D, po, F, n, Fn, Vn, nn, V, Q);
    }
}
#define TD_DISPATCH(fn, ...)                                                                  \
    switch (h->m.cost_kind) {                                                                 \
    case SDPB_COST_BACKORDER: fn<SDPB_COST_BACKORDER>(__VA_ARGS__); break;                    \
    case SDPB_COST_CASH_DEPOSIT: fn<SDPB_COST_CASH_DEPOSIT>(__VA_ARGS__); break;              \
    case SDPB_COST_CASH_OVERDRAFT: fn<SDPB_COST_CASH_OVERDRAFT>(__VA_ARGS__); break;          \
    case SDPB_COST_CASH_XR: fn<SDPB_COST_CASH_XR>(__VA_ARGS__); break;                        \
    case SDPB_COST_CASH_OD_LIMIT: fn<SDPB_COST_CASH_OD_LIMIT>(__VA_ARGS__); break;            \
    case SDPB_COST_CASH_OD_TESTING: fn<SDPB_COST_CASH_OD_TESTING>(__VA_ARGS__); break;        \
    default: fn<SDPB_COST_CASH_LOAN>(__VA_ARGS__); break;                                     \
    }

// N_t: the roots of period t and the successors of the n_src states `src` of period t - 1 (`off`: their action offsets,
// `pairs` (state, action) pairs), minus the states the handle already holds in period t; sorted, into *out.
//
// Scratch: three key buffers of `cap` keys (chunk candidates, sort output, merge output / new states) and the radix
// sort's temporary storage, together at most `budget` bytes.  A chunk must hold at least as many candidates as the
// period has new states so far (cap - nf >= nf), so the merges of a period cost at most twice its sorted candidates; a
// period whose new states pass half a buffer fails with SDPB_ERR_NOMEM instead of crawling on.
int td_new_states(sdpb_topdown* h, int t, const TDKey* src, long long n_src, const long long* off, long long pairs,
                  const std::vector<TDKey>& roots, TDKey** out, long long* n_out) {
    *out = nullptr;
    *n_out = 0;
    const long long nr = (long long)roots.size();
    if (pairs == 0 && nr == 0) return SDPB_OK;
    const int nd = h->P.nd(), D = t > 1 ? h->pmf_len[t - 2] : 1;
    const TDKey* Fo = h->mt.F[t - 1];
    const long long no = h->mt.nF[t - 1];
    cudaStream_t st = h->mt.stream;
    auto par = thrust::cuda::par.on(st);
    const long long cand = pairs * D + nr, key3 = 3 * (long long)sizeof(TDKey);
    const std::string per = "period " + std::to_string(t);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const long long budget = h->scratch_bytes > 0 ? h->scratch_bytes : (long long)(free_b / 2);
    auto sort_temp = [&](long long items, size_t& bytes) {
        cub::DoubleBuffer<TDKey> probe(nullptr, nullptr);
        return td_sort_nd(nd, nullptr, bytes, probe, items, st) == cudaSuccess;
    };
    long long cap = std::max(1ll, std::min(cand, budget / key3));
    size_t tmp_bytes = 0;
    if (!sort_temp(cap, tmp_bytes)) return td_fail(h, SDPB_ERR_CUDA, "sizing the sort");
    if (cap * key3 + (long long)tmp_bytes > budget) {  // the temporary storage shrinks with the item count
        cap = (budget - (long long)tmp_bytes) / key3;
        if (cap < 1 || !sort_temp(cap, tmp_bytes) || cap * key3 + (long long)tmp_bytes > budget)
            return td_fail(h, SDPB_ERR_NOMEM, per + ": a scratch budget of " + std::to_string(budget) +
                                                  " bytes does not hold the sort's temporary storage");
    }
    auto too_many = [&](long long nf) {
        return td_fail(h, SDPB_ERR_NOMEM,
                       per + " reaches at least " + std::to_string(nf) + " new states: more than a scratch budget of " +
                           std::to_string(budget) + " bytes (" + std::to_string(cap) +
                           " keys per buffer, at most half of them new states) can expand");
    };
    if (nr > cap) return too_many(nr);
    memo::DevBuf kb[3], tmp_b;
    for (auto& b : kb)
        if (!b.alloc((size_t)cap * sizeof(TDKey)))
            return td_fail(h, SDPB_ERR_NOMEM, "allocation of the expansion scratch failed (" + per + ")");
    if (!tmp_b.alloc(tmp_bytes)) return td_fail(h, SDPB_ERR_NOMEM, "allocation of the sort scratch failed (" + per + ")");
    TDKey* front = (TDKey*)kb[0].p;
    TDKey* x = (TDKey*)kb[1].p;
    TDKey* y = (TDKey*)kb[2].p;
    long long nf = 0;
    try {
        if (nr > 0) {  // the roots (sorted and unique) that period t does not hold yet
            if (cudaMemcpyAsync(y, roots.data(), (size_t)nr * sizeof(TDKey), cudaMemcpyHostToDevice, st) != cudaSuccess)
                return td_fail(h, SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
            nf = thrust::set_difference(par, y, y + nr, Fo, Fo + no, front, TDLess()) - front;
        }
        for (long long p = 0; p < pairs;) {
            const long long room = cap - nf;
            const long long np = std::min(pairs - p, room / D);
            if (np < 1 || nf > room) return too_many(nf);
            TD_DISPATCH(launch_expand, h, t - 1, src, n_src, off, p, np, x)
            if (cudaGetLastError() != cudaSuccess) return td_fail(h, SDPB_ERR_CUDA, "td_expand launch failed");
            long long m = thrust::remove_if(par, x, x + np * D, TDIsHole()) - x;
            cub::DoubleBuffer<TDKey> db(x, y);
            size_t tb = tmp_bytes;
            if (td_sort_nd(nd, tmp_b.p, tb, db, m, st) != cudaSuccess) return td_fail(h, SDPB_ERR_CUDA, "radix sort failed");
            TDKey* cur = db.Current();
            TDKey* alt = db.Alternate();
            m = thrust::unique(par, cur, cur + m, TDEq()) - cur;
            thrust::merge(par, front, front + nf, cur, cur + m, alt, TDLess());
            const long long nm = thrust::unique(par, alt, alt + nf + m, TDEq()) - alt;
            TDKey* old = front;
            if (no > 0) {  // keep only what period t does not hold yet
                nf = thrust::set_difference(par, alt, alt + nm, Fo, Fo + no, cur, TDLess()) - cur;
                front = cur;
                y = alt;
            } else {
                nf = nm;
                front = alt;
                y = cur;
            }
            x = old;
            p += np;
        }
    } catch (const std::exception& ex) {
        return td_fail(h, SDPB_ERR_CUDA, std::string("sort / merge: ") + ex.what());
    }
    if (nf == 0) return cudaStreamSynchronize(st) == cudaSuccess ? SDPB_OK : td_fail(h, SDPB_ERR_CUDA, "forward pass");
    if (!memo::alloc(*out, nf)) return td_fail(h, SDPB_ERR_NOMEM, "allocation of the states of " + per + " failed");
    *n_out = nf;
    if (cudaMemcpyAsync(*out, front, (size_t)nf * sizeof(TDKey), cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
        return td_fail(h, SDPB_ERR_CUDA, std::string("forward pass: ") + cudaGetErrorString(cudaGetLastError()));
    return SDPB_OK;
}

// The forward pass of an extension from period p: N_t for t = p .. T into the stage, and the evaluations and capped XR
// action sets of the new states.
int td_forward(sdpb_topdown* h, int p, const std::vector<std::vector<TDKey>>& roots, memo::Stage<TDTraits>& sg,
               double& evals, double& capped_total) {
    const int T = h->m.T;
    cudaStream_t st = h->mt.stream;
    auto par = thrust::cuda::par.on(st);
    memo::DevBuf cap_b, off_b;  // off_b: exclusive prefix sum of |A_t(s)| over N_t (n + 1 entries)
    if (!cap_b.alloc(sizeof(unsigned long long))) return td_fail(h, SDPB_ERR_NOMEM, "allocation failed");
    unsigned long long* d_capped = (unsigned long long*)cap_b.p;
    long long pairs = 0;
    for (int t = p; t <= T; t++) {
        const int k = t - 1;
        const int rc = td_new_states(h, t, t > p ? sg.N[k - 1] : nullptr, t > p ? sg.nN[k - 1] : 0,
                                     (const long long*)off_b.p, pairs, roots[k], &sg.N[k], &sg.nN[k]);
        if (rc != SDPB_OK) return rc;
        const long long n = sg.nN[k];
        pairs = 0;
        if (n == 0) continue;
        if (!off_b.alloc((size_t)(n + 1) * sizeof(long long))) return td_fail(h, SDPB_ERR_NOMEM, "allocation of the action counts failed");
        long long* off = (long long*)off_b.p;
        if (cudaMemsetAsync(off, 0, sizeof(long long), st) != cudaSuccess ||
            cudaMemsetAsync(d_capped, 0, sizeof(unsigned long long), st) != cudaSuccess)
            return td_fail(h, SDPB_ERR_CUDA, "cudaMemsetAsync failed");
        TD_DISPATCH(launch_count, h, t, sg.N[k], n, off + 1, d_capped)
        unsigned long long capped = 0;
        try {
            thrust::inclusive_scan(par, off + 1, off + 1 + n, off + 1);
        } catch (const std::exception& ex) {
            return td_fail(h, SDPB_ERR_CUDA, std::string("scan: ") + ex.what());
        }
        if (cudaMemcpyAsync(&pairs, off + n, sizeof pairs, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaMemcpyAsync(&capped, d_capped, sizeof capped, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            return td_fail(h, SDPB_ERR_CUDA, std::string("counting the actions: ") + cudaGetErrorString(cudaGetLastError()));
        capped_total += (double)capped;
        evals += (double)pairs * h->pmf_len[k];
    }
    return SDPB_OK;
}

// getExpectedValue on the states roots[t - 1] of every period t >= p (each sorted and unique; roots[t - 1] empty for
// t < p): the forward pass builds the states no earlier call reached, the backward pass solves only those against the
// merged tables of the next period, and the merged tables of every touched period replace the handle's at the end.
int td_extend(sdpb_topdown* h, int p, const std::vector<std::vector<TDKey>>& roots) {
    memo::Stage<TDTraits> sg(h->m.T);
    if (cudaEventRecord(h->mt.e0, h->mt.stream) != cudaSuccess) return td_fail(h, SDPB_ERR_CUDA, "cudaEventRecord failed");
    double evals = 0, capped = 0;
    const int rc = td_forward(h, p, roots, sg, evals, capped);
    if (rc != SDPB_OK) return rc;
    if (capped > 0 && !(h->allow & SDPB_ALLOW_CAPPED_ACTIONS))
        return td_fail(h, SDPB_ERR_OFFGRID,
                       std::to_string((long long)capped) +
                           " reached XR states have an order-up-to range longer than max_order_idx + 1 "
                           "(allow SDPB_ALLOW_CAPPED_ACTIONS to cut it there)");
    auto backward = [h](int t, const TDKey* F, long long n, const TDKey* Fn, const double* Vn, long long nn, double* V,
                        int* Q) {
        TD_DISPATCH(launch_backward, h, t, F, n, Fn, Vn, nn, V, Q)
        return 1;
    };
    return memo::commit(h->mt, sg, p, evals, capped, backward, h->err);
}

template <int KIND>
int td_rollout(sdpb_topdown* h, const TDKey& k0, const double* samples, int n, double discount, double* values) {
    auto extend = [h](int p, const std::vector<std::vector<TDKey>>& r) { return td_extend(h, p, r); };
    return memo::rollout(h->mt, TDStep<KIND>{h->P}, k0, samples, n, 1, discount, extend, values, h->err);
}

// The key of one API-order state
TDKey td_key_of(const sdpb_topdown* h, const double* s) {
    int c = 1;
    const double w = h->P.cash ? s[c++] : 0.0;
    const double q1 = h->P.lead >= 1 ? s[c++] : 0.0;
    const double q2 = h->P.lead >= 2 ? s[c++] : 0.0;
    return td_pack(h->P, s[0], q1, q2, w);
}

// n API-order states -> their keys, sorted and unique; SDPB_ERR_ARG when a coordinate is not finite
int td_root_keys(sdpb_topdown* h, const double* states, int n, std::vector<TDKey>& out) {
    out.resize((size_t)n);
    for (int i = 0; i < n; i++) {
        const double* s = states + (size_t)i * h->ndim;
        for (int k = 0; k < h->ndim; k++)
            if (!std::isfinite(s[k])) return td_fail(h, SDPB_ERR_ARG, "a state is not finite");
        out[i] = td_key_of(h, s);
    }
    memo::canonical<TDTraits>(out);
    return SDPB_OK;
}

void td_destroy(sdpb_topdown* h) {
    if (!h) return;
    if (h->device >= 0) cudaSetDevice(h->device);
    for (void* p : h->owned) cudaFree(p);
    delete h;  // and its memo tables
}

}  // namespace

extern "C" {

const char* sdpb_topdown_last_error(const sdpb_topdown* h) { return h ? h->err.c_str() : g_td_error.c_str(); }

void sdpb_topdown_destroy(sdpb_topdown* h) { td_destroy(h); }

int sdpb_topdown_solve(const sdpb_model* m, const sdpb_topdown_options* opt, const double* init_states, int n,
                       sdpb_topdown** out) {
    g_td_error.clear();
    if (!m || !out || !init_states || n < 1) return td_fail(nullptr, SDPB_ERR_ARG, "null argument or n < 1");
    *out = nullptr;
    if (m->struct_size != sizeof(sdpb_model)) return td_fail(nullptr, SDPB_ERR_ARG, "sdpb_model.struct_size does not match this library");
    if (opt && opt->struct_size != sizeof(sdpb_topdown_options))
        return td_fail(nullptr, SDPB_ERR_ARG, "sdpb_topdown_options.struct_size does not match this library");
    if (opt && opt->scratch_bytes < 0) return td_fail(nullptr, SDPB_ERR_ARG, "scratch_bytes < 0");
    if (m->T < 1 || !m->pmf_len || !m->pmf_d || !m->pmf_p) return td_fail(nullptr, SDPB_ERR_ARG, "T < 1 or null pmf");
    if (m->cost_kind == SDPB_COST_CASH_TWO_PRODUCT || m->cost_kind == SDPB_COST_STAFF)
        return td_fail(nullptr, SDPB_ERR_ARG, "the two-product and workforce kinds tie their action pairs or pmf rows to "
                                              "the grid: solve them with sdpb_create");
    if (m->cost_kind < 0 || m->cost_kind > SDPB_COST_STAFF) return td_fail(nullptr, SDPB_ERR_ARG, "bad cost_kind");
    if (m->terminal_value)
        return td_fail(nullptr, SDPB_ERR_ARG, "terminal_value is tabulated on the grid and has no value at an off-grid state");
    if (m->lead_time < 0 || m->lead_time > 2) return td_fail(nullptr, SDPB_ERR_ARG, "lead_time must be 0, 1 or 2");
    if ((m->cost_kind >= SDPB_COST_CASH_OD_LIMIT || m->cost_kind == SDPB_COST_CASH_XR) && m->lead_time != 0)
        return td_fail(nullptr, SDPB_ERR_ARG, "this cost kind has no lead-time variant in the reference");
    if (m->recursion != SDPB_REC_EXPECT && m->recursion != SDPB_REC_SURVIVAL) return td_fail(nullptr, SDPB_ERR_ARG, "bad recursion");
    if (m->recursion == SDPB_REC_SURVIVAL && !(m->cost_kind == SDPB_COST_CASH_DEPOSIT || m->cost_kind == SDPB_COST_CASH_OVERDRAFT))
        return td_fail(nullptr, SDPB_ERR_ARG, "survival recursion needs a cash kind");
    if (m->direction != SDPB_MIN && m->direction != SDPB_MAX) return td_fail(nullptr, SDPB_ERR_ARG, "bad direction");
    if (m->max_order_idx < 0) return td_fail(nullptr, SDPB_ERR_ARG, "max_order_idx < 0");
    if (!(m->step > 0) || !std::isfinite(m->step)) return td_fail(nullptr, SDPB_ERR_ARG, "step must be positive");
    if (has_cash(*m)) {
        if (!(m->q_mul > 0) || !(m->q_div > 0) || !(m->cash_max >= m->cash_min))
            return td_fail(nullptr, SDPB_ERR_ARG, "bad cash bounds or quantiser (q_mul, q_div > 0; cash_max >= cash_min)");
        if (m->quantiser == SDPB_Q_LONGDIV && (m->q_div != std::floor(m->q_div) || m->q_div < 1 || m->q_div > 9e18))
            return td_fail(nullptr, SDPB_ERR_ARG, "SDPB_Q_LONGDIV needs an integer q_div >= 1");
        if (m->quantiser != SDPB_Q_DIV && m->quantiser != SDPB_Q_LONGDIV && m->quantiser != SDPB_Q_TRUNC)
            return td_fail(nullptr, SDPB_ERR_ARG, "bad quantiser");
    }
    const int T = m->T;
    std::vector<int> len(m->pmf_len, m->pmf_len + T), poff(T + 1, 0);
    for (int t = 0; t < T; t++) {
        if (len[t] < 1) return td_fail(nullptr, SDPB_ERR_ARG, "empty pmf row");
        poff[t + 1] = poff[t] + len[t];
    }

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return td_fail(nullptr, SDPB_ERR_NO_DEVICE, "no CUDA device (libsdpb200 has no CPU path)");
    }
    int dev = opt ? opt->device : -1;
    if (dev < 0) cudaGetDevice(&dev);
    int cc_major = 0;
    if (dev >= ndev || cudaSetDevice(dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
        return td_fail(nullptr, SDPB_ERR_NO_DEVICE, "cannot select the CUDA device");
    if (cc_major != 10) return td_fail(nullptr, SDPB_ERR_NO_DEVICE, "libsdpb200 is built for sm_100a (B200) only");

    sdpb_topdown* h = new (std::nothrow) sdpb_topdown();
    if (!h) return td_fail(nullptr, SDPB_ERR_NOMEM, "out of host memory");
    h->m = *m;
    h->device = dev;
    h->allow = opt ? opt->allow : 0;
    h->scratch_bytes = opt ? opt->scratch_bytes : 0;
    h->pmf_len = len;
    h->pmf_off = poff;
    h->ndim = 1 + (has_cash(*m) ? 1 : 0) + m->lead_time;
    auto bail = [&](int rc, std::string msg) { td_destroy(h); return td_fail(nullptr, rc, msg); };
    if (h->mt.open(T, h->err) != SDPB_OK) return bail(SDPB_ERR_CUDA, h->err);

    // device model: the scalars the lambdas read, per-period tables expanded to T entries
    const int NP = poff[T];
    std::vector<double> pd(m->pmf_d, m->pmf_d + NP), pp(m->pmf_p, m->pmf_p + NP), pg(NP);
    for (int j = 0; j < NP; j++) pg[j] = pp[j] * m->gamma;  // first product of `p * gamma * V` (CashRecursion.java:120)
    std::vector<double> price_t(T), v_t(T), ovh_t(T), res_t(T);
    for (int t = 0; t < T; t++) {
        price_t[t] = m->price_t ? m->price_t[t] : m->price;
        v_t[t] = m->vari_cost_t ? m->vari_cost_t[t] : m->vari_cost;
        ovh_t[t] = m->overhead_t ? m->overhead_t[t] : m->overhead;
        res_t[t] = m->reserve_t ? m->reserve_t[t] : 0.0;
    }
    auto up = [&](const std::vector<double>& v) -> const double* {
        void* p = nullptr;
        if (cudaMalloc(&p, v.size() * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        h->owned.push_back(p);
        if (cudaMemcpyAsync(p, v.data(), v.size() * sizeof(double), cudaMemcpyHostToDevice, h->mt.stream) != cudaSuccess) return nullptr;
        return (const double*)p;
    };
    DevModel& d = h->P.M;
    d.cost_kind = m->cost_kind;
    d.recursion = m->recursion;
    d.is_min = (m->recursion == SDPB_REC_SURVIVAL) ? 0 : (m->direction == SDPB_MIN);
    d.T = T;
    d.lead = m->lead_time;
    d.max_order_idx = m->max_order_idx;
    d.flags = m->flags;
    d.quantiser = m->quantiser;
    d.nI = d.nQ = d.nW = 1;  // no grid
    d.inv_min = m->inv_min;
    d.step = m->step;
    d.cash_min = m->cash_min;
    d.cash_max = m->cash_max;
    d.q_mul = has_cash(*m) ? m->q_mul : 1.0;
    d.q_div = has_cash(*m) ? m->q_div : 1.0;
    d.q_idiv = (long long)d.q_div;
    d.K = m->fixed_cost;
    d.h = m->hold_cost;
    d.pen = m->penalty_cost;
    d.salvage = m->salvage;
    d.one_plus_dr = 1 + m->deposit_rate;
    d.one_minus_rho = 1 - m->overhead_rate;
    d.neg_r0 = -m->r0;
    d.r2 = m->r2;
    d.r3 = m->r3;
    d.od_limit = m->od_limit;
    d.interest_free = m->interest_free;
    d.r2_limit_term = m->r2 * (m->od_limit - m->interest_free);
    d.reserve2 = m->reserve2;
    d.dr = m->deposit_rate;
    d.q_from_period = m->q_from_period;
    d.price_t = up(price_t);
    d.v_t = up(v_t);
    d.ovh_t = up(ovh_t);
    d.reserve_t = up(res_t);
    d.pmf_d = up(pd);
    d.pmf_p = up(pp);
    d.pmf_pg = up(pg);
    if (!d.price_t || !d.v_t || !d.ovh_t || !d.reserve_t || !d.pmf_d || !d.pmf_p || !d.pmf_pg)
        return bail(SDPB_ERR_NOMEM, "allocation of the model tables failed");
    h->P.inv_max = m->inv_max;
    h->P.lead = m->lead_time;
    h->P.cash = has_cash(*m) ? 1 : 0;

    std::vector<std::vector<TDKey>> roots((size_t)T);
    int rc = td_root_keys(h, init_states, n, roots[0]);
    if (rc == SDPB_OK) rc = td_extend(h, 1, roots);
    if (rc != SDPB_OK) return bail(rc, h->err);
    *out = h;
    return SDPB_OK;
}

int sdpb_topdown_states(const sdpb_topdown* h, int64_t* n_states) {
    if (!h || !n_states) return SDPB_ERR_ARG;
    for (int t = 0; t < h->m.T; t++) n_states[t] = h->mt.nF[t];
    return SDPB_OK;
}

int sdpb_topdown_stats(const sdpb_topdown* h, sdpb_stats* s) {
    if (!h || !s) return SDPB_ERR_ARG;
    *s = h->mt.stats;
    return SDPB_OK;
}

int sdpb_topdown_value(sdpb_topdown* h, int period, const double* states, int n, double* v, double* q) {
    if (!h) return td_fail(nullptr, SDPB_ERR_ARG, "null handle");
    if (period < 1 || period > h->m.T || n < 0 || (n > 0 && !states)) return td_fail(h, SDPB_ERR_ARG, "bad period or states");
    if (n == 0) return SDPB_OK;
    cudaSetDevice(h->device);
    std::vector<TDKey> keys((size_t)n);
    for (int i = 0; i < n; i++) keys[i] = td_key_of(h, states + (size_t)i * h->ndim);
    std::vector<double> vv;
    std::vector<int> qi;
    const int rc = memo::lookup(h->mt, period, keys, vv, qi, h->err);
    if (rc != SDPB_OK) return rc;
    for (int i = 0; i < n; i++) {
        if (v) v[i] = vv[i];
        // bestOrderQty stays 0 when no action improves on the initial value; XR reports the order-up-to level
        const double a = qi[i] < 0 ? 0.0 : qi[i] * h->m.step;
        if (q) q[i] = (qi[i] >= 0 && h->m.cost_kind == SDPB_COST_CASH_XR) ? states[(size_t)i * h->ndim] + a : a;
    }
    return SDPB_OK;
}

int sdpb_topdown_opt_table(sdpb_topdown* h, double* rows, size_t* nrows) {
    if (!h || !nrows) return td_fail(h, SDPB_ERR_ARG, "null argument");
    cudaSetDevice(h->device);
    auto row = [h](int t, const TDKey& k, double, int qi, double* row) {
        double x, q1, q2, cw;
        td_unpack(h->P, k, x, q1, q2, cw);
        int c = 0;
        row[c++] = t;
        row[c++] = x;
        if (h->P.cash) row[c++] = cw;
        if (h->P.lead >= 1) row[c++] = q1;
        if (h->P.lead >= 2) row[c++] = q2;
        const double a = qi < 0 ? 0.0 : qi * h->m.step;
        row[c] = (qi >= 0 && h->m.cost_kind == SDPB_COST_CASH_XR) ? x + a : a;
    };
    return memo::opt_table(h->mt, rows, nrows, h->ndim + 2, row, h->err);
}

int sdpb_topdown_extend(sdpb_topdown* h, int period, const double* states, int n) {
    if (!h) return td_fail(nullptr, SDPB_ERR_ARG, "null handle");
    if (period < 1 || period > h->m.T || n < 0 || (n > 0 && !states)) return td_fail(h, SDPB_ERR_ARG, "bad period or states");
    if (n == 0) return SDPB_OK;
    std::vector<std::vector<TDKey>> roots((size_t)h->m.T);
    const int rc = td_root_keys(h, states, n, roots[period - 1]);
    if (rc != SDPB_OK) return rc;
    cudaSetDevice(h->device);
    return td_extend(h, period, roots);
}

int sdpb_topdown_simulate(sdpb_topdown* h, const double* init_state, const double* samples, int n, double discount,
                          double* values) {
    if (!h) return td_fail(nullptr, SDPB_ERR_ARG, "null handle");
    if (!init_state || !samples || !values || n < 1) return td_fail(h, SDPB_ERR_ARG, "null argument or n < 1");
    const int T = h->m.T;
    for (size_t i = 0; i < (size_t)n * T; i++)
        if (!std::isfinite(samples[i])) return td_fail(h, SDPB_ERR_ARG, "a sample is not finite");
    std::vector<std::vector<TDKey>> roots((size_t)T);
    int rc = td_root_keys(h, init_state, 1, roots[0]);
    if (rc != SDPB_OK) return rc;
    cudaSetDevice(h->device);
    TD_DISPATCH(rc = td_rollout, h, roots[0][0], samples, n, discount, values)
    return rc;
}

}  // extern "C"
