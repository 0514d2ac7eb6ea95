// kernel_cash.cuh — backward induction for the cash-constrained family (CashConstraint.java:95-133,
// cashSurvival.java:102-147 lambdas; CashRecursion.java:98-138 / RiskRecursion.java:66-104 loops) when
// every cash quantity is an exact integer.  Bit-identical to bi_generic by construction.
//
// Conditions (checked on the host, plan_cash): unit grid step, integer price / unit cost / fixed cost /
// overhead / cash bounds, no deposit interest, no overhead rate, no holding cost, no end-cash penalty,
// identity quantiser (round(w*1)/1), lost sales, consecutive integer demands.  Then, for t < T,
//     c(s,a,d) = price*min(x+a,d) - (K 1[a>0] + v a + overhead)
// and every intermediate of the reference's expression (revenue, deposit, the running differences,
// w + c, its clamp and Math.round) is an exactly representable integer, so
//   * the immediate value is F_j(y) - C_a with F_j(y) = price*min(y,d_j): ONE fp64 subtract, the same
//     for every cash level w — a thread owns R cash levels and shares it (and p_j * c) among them;
//   * the successor's cash index is iw + (F_j - C_a) clamped, in the integer ALU: no fp64 clamp, no
//     floor, no double->int conversion;
//   * once d_j >= y the sale is y units whatever the demand: successor and immediate value are
//     constant over the rest of the demand loop, so V_{t+1} is read once for all of those j.
// Per evaluation that leaves 3 + 2/R fp64 instructions (mul, add, add) and one coalesced 8-byte
// gather of V_{t+1} (lanes hold consecutive cash levels).  In the last period there is no successor:
// c = (exact integer part) + salvage*max(level,0) is shared by the R cash levels.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <vector>

#include "dev_model.cuh"
#include "kernel_generic.cuh"  // decode_state, prep_action, jmax0 / jmin
#include "kernel_lead.cuh"  // lds_double, lds_double2

namespace sdpb {

constexpr int kCashThreads = 64;
constexpr int kCashR = 4;                             // cash levels per thread
constexpr int kCashTile = kCashThreads * kCashR;      // cash levels per CTA

struct CashPeriod {
    bool ok = false;
    int price = 0, v = 0, ovh = 0, d0 = 0;
};

struct CashPlan {
    bool available = false;
    const char* why_not = "";
    int K = 0;
    std::vector<CashPeriod> period;
    // bi_cash_diag with the action range cut into slices (gridDim.z): per slice and state the slice's optimum,
    // merged by merge_action_slices.  Owned by the handle (allocated on first use from its pool).
    double* slice_v = nullptr;
    int* slice_a = nullptr;
    size_t slice_cap = 0;  // entries
};

struct CashArgs {
    int t, D, pmf_off;
    const double* Vn;
    double* Vt;
    int* Qt;
    long long lo, hi;
    int ix0;                     // first inventory row of the shard
    int price, v, K, ovh, d0, inv_min_i;
    double* slice_v;             // [gridDim.z][hi - lo] when the action range is sliced over gridDim.z
    int* slice_a;
};

// R cash levels per thread.  With a successor (t < T) every level gathers its own V_{t+1} entry and R = 4; in the
// last period there is no gather, the levels of a thread share c and p*c and differ only in their own running sum,
// so R = 16 brings the fp64 work down to 1 + 4/16 instructions per evaluation (R = 4: 7.8 ms of the 12 periods of C3).
constexpr int kCashRLast = 16;

template <bool SURVIVAL, bool IS_MIN, bool LAST, int R = kCashR>
__global__ void __launch_bounds__(kCashThreads)
bi_cash_int(const __grid_constant__ DevModel M, const __grid_constant__ CashArgs a) {
    constexpr int kCashTile = kCashThreads * R;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* PP = reinterpret_cast<double2*>(smem_raw);                          // (p, p*gamma)
    double* PRd = reinterpret_cast<double*>(smem_raw + (size_t)a.D * 16);        // price * d_j
    int* PRi = reinterpret_cast<int*>(smem_raw + (size_t)a.D * 24);              // same, as int
    for (int j = threadIdx.x; j < a.D; j += kCashThreads) {
        PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
        const int pr = a.price * (a.d0 + j);
        PRi[j] = pr;
        PRd[j] = (double)pr;
    }
    __syncthreads();

    const int ix = a.ix0 + blockIdx.x;
    const int iw0 = blockIdx.y * kCashTile + threadIdx.x;
    const double v_d = M.v_t[a.t - 1];
    const double res = M.reserve_t[a.t - 1];

    int iw[R], nA[R], arg[R];
    double best[R], wd[R];
    bool valid[R];
    int nAmax = 0;
#pragma unroll
    for (int r = 0; r < R; r++) {
        iw[r] = iw0 + r * kCashThreads;
        const long long idx = (long long)ix * M.nW + iw[r];
        valid[r] = iw[r] < M.nW && idx >= a.lo && idx < a.hi;
        iw[r] = min(iw[r], M.nW - 1);
        const double w = (double)(M.kmin + iw[r]);
        wd[r] = w;
        int n = M.max_order_idx + 1;
        if (M.flags & SDPB_F_CASH_LIMITED_ACTIONS) {  // CashConstraint.java:96-99
            const double bound = fmax(0.0, ((w - res) - M.reserve2) / v_d);
            n = (int)fmin((double)M.max_order_idx, bound) + 1;
        }
        nA[r] = valid[r] ? n : 0;
        nAmax = max(nAmax, nA[r]);
        best[r] = IS_MIN ? DBL_MAX : -DBL_MAX;
        arg[r] = kNoAction;
    }

    const int nW1 = M.nW - 1;
    // action slices over gridDim.z, as in bi_cash_diag: a band of the grid (one shard of eight) is a few hundred CTAs of
    // two warps, each a serial loop over ~200 actions x 200 demands -- the slices make that 16 times as many CTAs
    const int parts = (int)gridDim.z, part = (int)blockIdx.z;
    const int per_part = (nAmax + parts - 1) / parts;
    const int ai_end = min(nAmax, (part + 1) * per_part);
    for (int ai = part * per_part; ai < ai_end; ai++) {
        const int yv = a.inv_min_i + ix + ai;                 // stock after ordering, as a value
        const int CI = (ai > 0 ? a.K : 0) + a.v * ai + a.ovh;  // K 1[a>0] + v a + overhead
        const double Cd = (double)CI;
        const int jy = min(max(yv - a.d0, 0), a.D);          // demands d_j < y  <=>  j < jy
        double acc[R];
#pragma unroll
        for (int r = 0; r < R; r++) acc[r] = 0.0;

        if (LAST) {
            // terminal period: no successor.  c = exact integer part + salvage * max(level, 0)
            // (CashConstraint.java:112-113); the survival recursion scores 1[w + c >= 0]
            // (RiskRecursion.java:80-84).
            for (int j = 0; j < a.D; j++) {
                const double2 pp = PP[j];
                double c;
                if (j < jy) c = (PRd[j] - Cd) + M.salvage * (double)(yv - (a.d0 + j));
                else c = ((double)(a.price * yv) - Cd) + M.salvage * 0.0;
                if (!SURVIVAL) {
                    const double m = pp.x * c;
#pragma unroll
                    for (int r = 0; r < R; r++) acc[r] += m;
                } else {
#pragma unroll
                    for (int r = 0; r < R; r++) acc[r] += pp.x * ((wd[r] + c) >= 0.0 ? 1.0 : 0.0);
                }
            }
        } else {
        // ---- demand below the stock: sale = d_j, successor inventory y - d_j > 0 ----
            // All index arithmetic is 32-bit (plan_cash checks nI*nW < 2^31): the successor's flat index
            // is clamp(rowoff + iw + shift, rowoff, rowoff + nW-1), one add-max and one min per level.
#pragma unroll 2
            for (int j = 0; j < jy; j++) {
                const double2 pp = PP[j];
                int il = ix + ai - (a.d0 + j);                    // successor inventory index
                il = min(il, M.nI - 1);
                il = max(il, 0);
                const int rowoff = il * M.nW;
                const int kk0 = rowoff + PRi[j] - CI;             // + iw[r] = unclamped flat index
                const int khi = rowoff + nW1;
                double m = 0.0;
                if (!SURVIVAL) m = pp.x * (PRd[j] - Cd);          // p_j * c(s,a,d_j)
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int k = min(max(kk0 + iw[r], rowoff), khi);  // clamp to [cash_min, cash_max]
                    double vn = __ldg(a.Vn + (unsigned)k);
                    if (SURVIVAL && k - rowoff < -M.kmin) vn = 0.0;  // successor cash < 0: RiskRecursion.java:87-95
                    if (!SURVIVAL) acc[r] += m;                    // CashRecursion.java:117
                    acc[r] += pp.y * vn;                           // CashRecursion.java:120
                }
            }
            // ---- stock-out: sale = y for every remaining demand, successor inventory 0 ----
            if (jy < a.D) {
                const int PYi = a.price * yv;
                const int il = min(max(M.i_zero, 0), M.nI - 1);
                const int rowoff = il * M.nW;
                const int kk0 = rowoff + PYi - CI;
                const int khi = rowoff + nW1;
                const double inc = (double)PYi - Cd;
                double vn[R];
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int k = min(max(kk0 + iw[r], rowoff), khi);
                    vn[r] = __ldg(a.Vn + (unsigned)k);
                    if (SURVIVAL && k - rowoff < -M.kmin) vn[r] = 0.0;
                }
#pragma unroll 2
                for (int j = jy; j < a.D; j++) {
                    const double2 pp = PP[j];
                    double m = 0.0;
                    if (!SURVIVAL) m = pp.x * inc;
#pragma unroll
                    for (int r = 0; r < R; r++) {
                        if (!SURVIVAL) acc[r] += m;
                        acc[r] += pp.y * vn[r];
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (ai < nA[r] && (IS_MIN ? (acc[r] < best[r]) : (acc[r] > best[r]))) { best[r] = acc[r]; arg[r] = ai; }
        }
    }
    const long long n_local = a.hi - a.lo;
#pragma unroll
    for (int r = 0; r < R; r++) {
        if (valid[r]) {
            const long long idx = (long long)ix * M.nW + iw[r];
            if (parts == 1) {
                a.Vt[idx] = best[r];
                a.Qt[idx] = arg[r] == kNoAction ? -1 : arg[r];
            } else {  // merge_action_slices picks the first optimum over the slices
                a.slice_v[(long long)part * n_local + (idx - a.lo)] = best[r];
                a.slice_a[(long long)part * n_local + (idx - a.lo)] = arg[r];
            }
        }
    }
}

// ---- host side --------------------------------------------------------------------------------
inline bool cash_is_small_int(double x, double lim = 1048576.0) { return x == std::floor(x) && std::fabs(x) < lim; }

inline void plan_cash(CashPlan& P, const sdpb_model& m, const DevModel& d, const std::vector<int>& pmf_len,
                      const std::vector<int>& pmf_off, const std::vector<int>& pdi) {
    P.available = false;
    P.period.assign(m.T, CashPeriod{});
    if (m.cost_kind != SDPB_COST_CASH_DEPOSIT) { P.why_not = "only the deposit cash kind"; return; }
    if (m.lead_time != 0) { P.why_not = "lead time"; return; }
    if (m.step != 1.0) { P.why_not = "step != 1"; return; }
    if (!(m.flags & SDPB_F_LOST_SALES) || !(m.flags & SDPB_F_CLAMP_INV)) { P.why_not = "needs lost sales + clamp"; return; }
    if (m.q_mul != 1.0 || m.q_div != 1.0) { P.why_not = "quantiser is not round(w*1)/1"; return; }
    if (m.deposit_rate != 0.0 || m.overhead_rate != 0.0 || m.penalty_cost != 0.0 || m.hold_cost != 0.0) {
        P.why_not = "deposit rate, overhead rate, penalty and holding cost must be 0";
        return;
    }
    if (!cash_is_small_int(m.fixed_cost) || !cash_is_small_int(m.cash_min) || !cash_is_small_int(m.cash_max) ||
        !cash_is_small_int(m.inv_min) || m.inv_min < 0) { P.why_not = "non-integer parameters"; return; }
    P.K = (int)m.fixed_cost;
    bool any = false;
    for (int t = 0; t < m.T; t++) {
        const double price = m.price_t ? m.price_t[t] : m.price;
        const double v = m.vari_cost_t ? m.vari_cost_t[t] : m.vari_cost;
        const double ovh = m.overhead_t ? m.overhead_t[t] : m.overhead;
        if (!cash_is_small_int(price, 32768) || !cash_is_small_int(v, 32768) || !cash_is_small_int(ovh) || v <= 0) continue;
        const int* di = pdi.data() + pmf_off[t];
        bool consec = true;
        for (int j = 0; j < pmf_len[t]; j++) consec = consec && di[j] == di[0] + j;
        if (!consec) continue;
        // magnitude guard: every integer stays far inside int32
        const double big = std::fabs(price) * (std::fabs(m.inv_max) + d.max_order_idx + std::abs(di[0]) + pmf_len[t]) +
                           std::fabs(m.cash_min) + std::fabs(m.cash_max) + std::fabs(v) * d.max_order_idx +
                           std::fabs(m.fixed_cost) + std::fabs(ovh);
        if (big > 5e8 || (double)d.nI * d.nW > 2.0e9) continue;
        CashPeriod& cp = P.period[t];
        cp.ok = true;
        cp.price = (int)price; cp.v = (int)v; cp.ovh = (int)ovh; cp.d0 = di[0];
        any = true;
    }
    if (!any) { P.why_not = "no period qualifies"; return; }
    P.available = true;
}

// Shape of a bi_cash_int launch over [lo, hi): R = 16 cash levels per thread in the last period when the grid is large
// enough, and the action range cut into slices when the launch would otherwise leave the GPU short of CTAs.  gridDim.y
// = ceil(nW / tile) stays far below CUDA's 65535: plan_cash keeps |cash_min| and |cash_max| below 2^20, so nW < 2^21
// and the y dimension is at most 8192.
struct CashIntShape { bool wide; int tile, parts; dim3 grid; };

inline CashIntShape cash_int_shape(const sdpb_model& m, const DevModel& dm, int t, long long lo, long long hi, int sm_count) {
    CashIntShape s;
    const int rows = (int)((hi - 1) / dm.nW) - (int)(lo / dm.nW) + 1;
    const bool surv = m.recursion == SDPB_REC_SURVIVAL;
    const long long want = 64LL * sm_count;  // CTAs of two warps: ~8 resident per SM, 8 rounds of them
    const int max_parts = std::max(1, std::min(16, (m.max_order_idx + 1) / 12));
    auto parts_for = [&](long long tiles) {
        return tiles >= want ? 1 : (int)std::min<long long>((want + tiles - 1) / tiles, max_parts);
    };
    const long long tiles16 = (long long)rows * ((dm.nW + kCashThreads * kCashRLast - 1) / (kCashThreads * kCashRLast));
    // 16 cash levels per thread in the last period when the action slices still leave two CTAs per SM
    s.wide = t == m.T && !surv && dm.nW >= kCashThreads * kCashRLast / 2 && tiles16 * parts_for(tiles16) >= 2LL * sm_count;
    s.tile = kCashThreads * (s.wide ? kCashRLast : kCashR);
    const long long tiles = (long long)rows * ((dm.nW + s.tile - 1) / s.tile);
    s.parts = parts_for(tiles);
    if (s.wide && tiles16 >= 3LL * sm_count) s.parts = 1;  // measured on C3 (1002 CTAs): 103.9 ms unsliced, 104.6 in 10 slices
    s.grid = dim3((unsigned)rows, (unsigned)((dm.nW + s.tile - 1) / s.tile), (unsigned)s.parts);
    return s;
}

inline size_t cash_int_smem(int D) { return (size_t)D * 28 + 16; }

// For a period with a plan and cash_int_smem(D) <= 200 KB.  SDPB_OK, SDPB_ERR_NOMEM (slice scratch too small: the caller
// sizes it with sh = cash_int_shape) or SDPB_ERR_CUDA.
inline int launch_cash(const CashPlan& P, const CashIntShape& sh, const sdpb_model& m, const DevModel& dm, int t, int D,
                       int pmf_off, const double* Vn, double* Vt, int* Qt, long long lo, long long hi, cudaStream_t stream,
                       const DevPeer* d_peers, int n_peers) {
    if (hi <= lo) return SDPB_OK;
    const CashPeriod& cp = P.period[t - 1];
    CashArgs a;
    a.t = t; a.D = D; a.pmf_off = pmf_off; a.Vn = Vn; a.Vt = Vt; a.Qt = Qt; a.lo = lo; a.hi = hi;
    a.ix0 = (int)(lo / dm.nW);
    a.price = cp.price; a.v = cp.v; a.K = P.K; a.ovh = cp.ovh; a.d0 = cp.d0; a.inv_min_i = (int)m.inv_min;
    const bool surv = m.recursion == SDPB_REC_SURVIVAL;
    const bool wide = sh.wide;
    const dim3 grid = sh.grid;
    const long long n_local = hi - lo;
    if (sh.parts > 1) {
        if ((size_t)sh.parts * (size_t)n_local > P.slice_cap) return SDPB_ERR_NOMEM;
        a.slice_v = P.slice_v; a.slice_a = P.slice_a;
    } else { a.slice_v = nullptr; a.slice_a = nullptr; }
    const size_t smem = cash_int_smem(D);
    if (smem > 48 * 1024) {
        cudaFuncSetAttribute(bi_cash_int<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(bi_cash_int<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(bi_cash_int<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(bi_cash_int<false, true, true, kCashRLast>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(bi_cash_int<false, false, true, kCashRLast>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(bi_cash_int<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(bi_cash_int<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(bi_cash_int<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    if (t == m.T) {
        if (surv) bi_cash_int<true, false, true><<<grid, kCashThreads, smem, stream>>>(dm, a);
        else if (wide) {
            if (dm.is_min) bi_cash_int<false, true, true, kCashRLast><<<grid, kCashThreads, smem, stream>>>(dm, a);
            else bi_cash_int<false, false, true, kCashRLast><<<grid, kCashThreads, smem, stream>>>(dm, a);
        } else {
            if (dm.is_min) bi_cash_int<false, true, true><<<grid, kCashThreads, smem, stream>>>(dm, a);
            else bi_cash_int<false, false, true><<<grid, kCashThreads, smem, stream>>>(dm, a);
        }
    } else {
        if (surv) bi_cash_int<true, false, false><<<grid, kCashThreads, smem, stream>>>(dm, a);
        else if (dm.is_min) bi_cash_int<false, true, false><<<grid, kCashThreads, smem, stream>>>(dm, a);
        else bi_cash_int<false, false, false><<<grid, kCashThreads, smem, stream>>>(dm, a);
    }
    if (cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    if (sh.parts > 1) {
        const unsigned mb = (unsigned)((n_local + 255) / 256);
        if (dm.is_min && !surv) merge_action_slices<true><<<mb, 256, 0, stream>>>(P.slice_v, P.slice_a, sh.parts, n_local, Vt + lo, Qt + lo, lo, d_peers, n_peers, t);
        else merge_action_slices<false><<<mb, 256, 0, stream>>>(P.slice_v, P.slice_a, sh.parts, n_local, Vt + lo, Qt + lo, lo, d_peers, n_peers, t);
        if (cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    }
    return SDPB_OK;
}

// ---------------------------------------------------------------------------------------------
// bi_cash_diag — the same integer-exact model with a register window along the (1, -price) diagonal.
//
// For a fixed action a and demand d_j < y = x + a the successor is
//     ( level l = y - d_j ,  cash w + price*d_j - C_a )  =  ( l ,  [w + price*x] + price*a - C_a - price*l ),
// which depends on the state only through phi = w + price*x.  States (x+k, w - price*k) share phi, so
// slot k at demand j+1 needs exactly the value slot k-1 needed at demand j (the cash and inventory
// clamps are functions of the unclamped successor and therefore shared too), and once d_j >= y every
// slot's successor is the same stock-out entry (0, phi + price*a - C_a).  A thread owns YT = 8 such
// diagonal states for ALL actions (no cross-thread argopt at all); per demand point it gathers ONE new
// value (instead of 8), forms p_j*c once for all slots still in stock, and spends (add, mul, add) per
// evaluation: 3 + 2/8 fp64 instructions and 1/8 gather per evaluation (bi_cash_int: 3.5 and 1).
// Lanes hold consecutive cash levels, so every gather is a coalesced row segment.
// Demand steps split into: all slots in stock (fast path, window rotation unrolled x(YT+PF)) / mixed
// (per-slot select, the 7 steps between slot 0 and slot 7 stocking out) / all slots stocked out (no
// window, no loads).  64-thread CTAs, 8 per SM: the grid is only ~2000 CTAs on a 1e6-state model, so
// small CTAs are what keeps the last wave short (ncu: profiles/r01_ncu_cash_diag*_raw.csv).
constexpr int kDiagYT = 8;
constexpr int kDiagCols = 64;  // state columns (cash levels of slot 0) per CTA

template <bool SURVIVAL, bool IS_MIN>
__global__ void __launch_bounds__(kDiagCols, 512 / kDiagCols)
bi_cash_diag(const __grid_constant__ DevModel M, const __grid_constant__ CashArgs a) {
    constexpr int kDiagThreads = kDiagCols;
    constexpr int YT = kDiagYT, PF = 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* PP = reinterpret_cast<double2*>(smem_raw);                    // (p, p*gamma)
    double* PRd = reinterpret_cast<double*>(smem_raw + (size_t)a.D * 16);  // price * d_j
    for (int j = threadIdx.x; j < a.D; j += kDiagThreads) {
        PP[j] = make_double2(M.pmf_p[a.pmf_off + j], M.pmf_pg[a.pmf_off + j]);
        PRd[j] = (double)(a.price * (a.d0 + j));
    }
    __syncthreads();
    const unsigned pp_s = (unsigned)__cvta_generic_to_shared(PP);
    const unsigned pr_s = (unsigned)__cvta_generic_to_shared(PRd);
    // action split: gridDim.z CTAs share a tile of state columns and take one slice of the action range each.  The
    // grid of a 1e6-state model is only ~2000 CTAs of 2 warps -- 14 per SM, where one CTA more or less on an SM is a
    // 7 % tail, and 1.8 per SM on an eighth of the grid -- so the unit of work is made 4-16 times smaller and the
    // block scheduler balances the SMs; every slice writes its optimum per state and merge_action_slices picks
    // the first best one (ascending slices hold ascending actions).
    const int parts = (int)gridDim.z;
    const int part = (int)blockIdx.z, col = threadIdx.x;

    const int D = a.D, price = a.price, nW1 = M.nW - 1;
    const int ix0 = a.ix0 + blockIdx.y * YT;                                  // inventory index of slot 0
    const int iw0 = blockIdx.x * kDiagCols + col;                             // cash index of slot 0
    const double v_d = M.v_t[a.t - 1];
    const double res = M.reserve_t[a.t - 1];

    int nA[YT], arg[YT];
    double best[YT];
    int nAmax = 0;
#pragma unroll
    for (int k = 0; k < YT; k++) {
        const int iw = iw0 - price * k, ix = ix0 + k;
        const long long idx = (long long)ix * M.nW + iw;
        const bool valid = iw >= 0 && iw < M.nW && ix < M.nI && idx >= a.lo && idx < a.hi;
        int n = M.max_order_idx + 1;
        if (M.flags & SDPB_F_CASH_LIMITED_ACTIONS) {  // CashConstraint.java:96-99
            const double w = (double)(M.kmin + iw);
            const double bound = fmax(0.0, ((w - res) - M.reserve2) / v_d);
            n = (int)fmin((double)M.max_order_idx, bound) + 1;
        }
        nA[k] = valid ? n : 0;
        nAmax = max(nAmax, nA[k]);
        best[k] = IS_MIN ? DBL_MAX : -DBL_MAX;
        arg[k] = kNoAction;
    }
    if (nAmax == 0) return;

    const int xv0 = a.inv_min_i + ix0;  // inventory VALUE of slot 0
    const int row_tail = min(max(M.i_zero, 0), M.nI - 1) * M.nW;
    const int per_part = (nAmax + parts - 1) / parts;
    const int ai_end = min(nAmax, (part + 1) * per_part);

    for (int ai = part * per_part; ai < ai_end; ai++) {
        const int CI = (ai > 0 ? a.K : 0) + a.v * ai + a.ovh;  // K 1[a>0] + v a + overhead
        const double Cd = (double)CI;
        const int base = iw0 + price * (ix0 + ai) - CI;        // successor cash index = base - price*il
        const int L0 = ix0 + ai - a.d0;                        // slot k, demand j: level index L0 + k - j
        const int jy0 = min(max(xv0 + ai - a.d0, 0), D);       // slot 0 is in stock for j < jy0
        const int jy7 = min(max(xv0 + (YT - 1) + ai - a.d0, 0), D);
        // Window of W = YT + PF registers: at demand j (phase JJ = j mod W) slot k reads Vw[(k - JJ) mod W]; the PF
        // free entries hold the levels slot 0 reaches at j+1 .. j+PF (loaded earlier), so every load lands in its
        // final register PF + 1 steps ahead of its first use and nothing is ever moved.
        constexpr int W = YT + PF;
        double acc[YT], Vw[W];
#pragma unroll
        for (int k = 0; k < YT; k++) acc[k] = 0.0;

        // gather V_{t+1} at level index il.  Levels <= 0 are fetched too (address clamped into the grid) but
        // never used: a slot reads its window only while it is in stock.
        const int row_max = (M.nI - 1) * M.nW;
        auto gather_at = [&](int ro, int c) -> double {  // ro = il*nW, c = base - price*il, both unclamped
            const int row = max(min(ro, row_max), 0);    // upper clamp first, as in the reference
            const int kc = max(min(c, nW1), 0);
            double vn = __ldg(a.Vn + (unsigned)(row + kc));
            if (SURVIVAL && M.kmin + kc < 0) vn = 0.0;  // RiskRecursion.java:87-95
            return vn;
        };
#pragma unroll
        for (int k = 0; k < W; k++) {
            const int il = k < YT ? L0 + k : L0 + k - W;  // entries YT..W-1: levels L0-PF .. L0-1
            Vw[k] = gather_at(il * M.nW, base - price * il);
        }
        // the entry slot 7 releases at demand j is reloaded with the level slot 0 reaches at demand j + 1 + PF
        int ro_run = (L0 - PF - 1) * M.nW, c_run = base - price * (L0 - PF - 1);

        int j = 0;
        // ---- all 8 slots in stock: shared p*c, one new gather per demand point ----
#define SDPB_DIAG_FAST(JJ)                                                                       \
        {                                                                                            \
            const double2 pp = lds_double2(pp_s + (unsigned)j * 16u);                                \
            double m = 0.0;                                                                          \
            if (!SURVIVAL) m = pp.x * (lds_double(pr_s + (unsigned)j * 8u) - Cd);  /* p_j * c */    \
            _Pragma("unroll") for (int k = 0; k < YT; k++) {                                         \
                if (!SURVIVAL) acc[k] += m;                        /* CashRecursion.java:117 */     \
                acc[k] += pp.y * Vw[(k - (JJ) + W) % W];           /* CashRecursion.java:120 */     \
            }                                                                                        \
            Vw[(YT - 1 - (JJ) + W) % W] = gather_at(ro_run, c_run);   /* slot 7's entry is free now */ \
            ro_run -= M.nW;                                                                          \
            c_run += price;                                                                          \
            j += 1;                                                                                  \
        }
        // The same step with the gather address taken from ONE running offset: inside a block of W steps the unclamped
        // row offset falls by nW and the unclamped cash index rises by price per step, so when no clamp changes state
        // inside the block -- rows inside the grid; cash either inside [0, nW-1] throughout or at/above the upper clamp
        // throughout -- the address is off0 + s*delta (delta = price - nW, or -nW under the upper cash clamp) and the
        // two clamps, two running adds and the combine of gather_at (7 integer instructions per step; the fp64 pipe
        // takes two dispatch slots per instruction, so every other instruction costs half an fp64 instruction:
        // ncu, profiles/r02_ncu_cash_diag.md) shrink to one add.
#define SDPB_DIAG_FAST_LIN(JJ)                                                                   \
        {                                                                                            \
            const double2 pp = lds_double2(pp_s + (unsigned)j * 16u);                                \
            const double m = pp.x * (lds_double(pr_s + (unsigned)j * 8u) - Cd);  /* p_j * c */      \
            _Pragma("unroll") for (int k = 0; k < YT; k++) {                                         \
                acc[k] += m;                                       /* CashRecursion.java:117 */     \
                acc[k] += pp.y * Vw[(k - (JJ) + W) % W];           /* CashRecursion.java:120 */     \
            }                                                                                        \
            Vw[(YT - 1 - (JJ) + W) % W] = __ldg(a.Vn + (unsigned)off_lin);                           \
            off_lin += delta_lin;                                                                    \
            j += 1;                                                                                  \
        }
        while (j + W <= jy0) {
            const int ro_last = ro_run - (W - 1) * M.nW, c_last = c_run + (W - 1) * price;  // (price > 0: cash_diag_ok)
            const bool rows_in = ro_last >= 0 && ro_run <= row_max;
            const bool cash_in = c_run >= 0 && c_last <= nW1, cash_hi = c_run >= nW1;
            if (!SURVIVAL && rows_in && (cash_in || cash_hi)) {
                int off_lin = ro_run + (cash_in ? c_run : nW1);
                const int delta_lin = cash_in ? price - M.nW : -M.nW;
#pragma unroll
                for (int JJ = 0; JJ < W; JJ++) SDPB_DIAG_FAST_LIN(JJ)
                ro_run -= W * M.nW;
                c_run += W * price;
            } else {
#pragma unroll
                for (int JJ = 0; JJ < W; JJ++) SDPB_DIAG_FAST(JJ)
            }
        }
#undef SDPB_DIAG_FAST_LIN
        // ---- stock-out entry: the same for every slot ----
        const int kt = min(max(iw0 + price * (xv0 + ai) - CI, 0), nW1);
        double Vtail = __ldg(a.Vn + (unsigned)(row_tail + kt));
        if (SURVIVAL && M.kmin + kt < 0) Vtail = 0.0;
        double inct[YT];  // price*y_k - C_a
#pragma unroll
        for (int k = 0; k < YT; k++) inct[k] = (double)(price * (xv0 + k + ai) - CI);
        // ---- remainder of the in-stock run (j < jy0), then the mixed region: some slots stocked out ----
        while (j < jy7) {
#pragma unroll
            for (int JJ = 0; JJ < W; JJ++) {
                if (j < jy0) SDPB_DIAG_FAST(JJ)
                else if (j < D) {
                    const double2 pp = lds_double2(pp_s + (unsigned)j * 16u);
                    const double cin = lds_double(pr_s + (unsigned)j * 8u) - Cd;
#pragma unroll
                    for (int k = 0; k < YT; k++) {
                        const bool in_stock = j < min(max(xv0 + k + ai - a.d0, 0), D);
                        if (!SURVIVAL) acc[k] += pp.x * (in_stock ? cin : inct[k]);
                        acc[k] += pp.y * (in_stock ? Vw[(k - JJ + W) % W] : Vtail);
                    }
                    Vw[(YT - 1 - JJ + W) % W] = gather_at(ro_run, c_run);
                    ro_run -= M.nW;
                    c_run += price;
                    j += 1;
                }
            }
        }
#undef SDPB_DIAG_FAST
        // ---- every slot stocked out: no window, no loads ----
        for (; j < D; j++) {
            const double2 pp = lds_double2(pp_s + (unsigned)j * 16u);
            const double pvt = pp.y * Vtail;
#pragma unroll
            for (int k = 0; k < YT; k++) {
                if (!SURVIVAL) acc[k] += pp.x * inct[k];
                acc[k] += pvt;
            }
        }
#pragma unroll
        for (int k = 0; k < YT; k++) {
            if (ai < nA[k] && (IS_MIN ? (acc[k] < best[k]) : (acc[k] > best[k]))) { best[k] = acc[k]; arg[k] = ai; }
        }
    }
    const long long n_local = a.hi - a.lo;
#pragma unroll
    for (int k = 0; k < YT; k++) {
        if (nA[k] > 0) {
            const long long idx = (long long)(ix0 + k) * M.nW + (iw0 - price * k);
            if (parts == 1) {
                a.Vt[idx] = best[k];
                a.Qt[idx] = arg[k] == kNoAction ? -1 : arg[k];
            } else {
                a.slice_v[(long long)part * n_local + (idx - a.lo)] = best[k];
                a.slice_a[(long long)part * n_local + (idx - a.lo)] = arg[k];
            }
        }
    }
}

// Slices of the action range for a launch over [lo, hi): up to 16, at least ~12 actions per slice.
inline int cash_diag_parts(const sdpb_model& m, const DevModel& dm, const CashPeriod& cp, long long lo, long long hi, int sm_count) {
    const int ix0 = (int)(lo / dm.nW), ix1 = (int)((hi - 1) / dm.nW);
    const int span_w = dm.nW + cp.price * (kDiagYT - 1);
    const long long tiles = (long long)((span_w + kDiagCols - 1) / kDiagCols) * ((ix1 - ix0 + 1 + kDiagYT - 1) / kDiagYT);
    const long long want = 256LL * sm_count;  // measured on C3: 3 slices 114.9 ms, 4: 113.7, 8: 111.5, 16: 110.2; an eighth of the grid: 4: 19.5, 8: 17.5, 16: 16.6
    int parts = 1;
    if (tiles < want) parts = (int)std::min<long long>((want + tiles - 1) / tiles, 16);
    parts = std::max(1, std::min(parts, (m.max_order_idx + 1) / 12));
    return parts;
}

inline size_t cash_diag_smem(int D) { return (((size_t)D * 24 + 15) & ~(size_t)15) + 16; }

// Whether bi_cash_diag can solve a period (t < T) whose integer plan is cp.  The launch puts the 8-row tiles on
// gridDim.y, which CUDA caps at 65535: a whole-grid bound, since no shard has more rows than the grid.
inline bool cash_diag_ok(const CashPeriod& cp, const sdpb_model& m, const DevModel& dm, int D) {
    return cp.price > 0 && cp.price * (kDiagYT - 1) <= dm.nW &&  // the diagonal must stay on the cash axis
           (long long)(dm.nI + D + std::abs(cp.d0) + 2 * kDiagYT + m.max_order_idx) * dm.nW < 0x7fffffffLL &&  // 32-bit row offsets
           (dm.nI + kDiagYT - 1) / kDiagYT <= 65535 &&
           cash_diag_smem(D) <= 200 * 1024;
}

// For a period t < T with a plan and cash_diag_ok; `parts` = cash_diag_parts.  SDPB_OK, SDPB_ERR_NOMEM or SDPB_ERR_CUDA.
inline int launch_cash_diag(const CashPlan& P, int parts, const sdpb_model& m, const DevModel& dm, int t, int D, int pmf_off,
                            const double* Vn, double* Vt, int* Qt, long long lo, long long hi, cudaStream_t stream,
                            const DevPeer* d_peers, int n_peers) {
    if (hi <= lo) return SDPB_OK;
    const CashPeriod& cp = P.period[t - 1];
    CashArgs a;
    a.t = t; a.D = D; a.pmf_off = pmf_off; a.Vn = Vn; a.Vt = Vt; a.Qt = Qt; a.lo = lo; a.hi = hi;
    a.ix0 = (int)(lo / dm.nW);
    const int ix1 = (int)((hi - 1) / dm.nW);
    a.price = cp.price; a.v = cp.v; a.K = P.K; a.ovh = cp.ovh; a.d0 = cp.d0; a.inv_min_i = (int)m.inv_min;
    const int span_w = dm.nW + cp.price * (kDiagYT - 1);  // slot 0's cash index runs past the axis so slot 7 covers it
    const unsigned gx = (unsigned)((span_w + kDiagCols - 1) / kDiagCols), gy = (unsigned)((ix1 - a.ix0 + 1 + kDiagYT - 1) / kDiagYT);
    const long long n_local = hi - lo;
    if (parts > 1) {
        const size_t need = (size_t)parts * (size_t)n_local;
        if (need > P.slice_cap) return SDPB_ERR_NOMEM;  // (the caller sizes the scratch)
        a.slice_v = P.slice_v; a.slice_a = P.slice_a;
        // (every slice writes every state of [lo, hi): a valid state has at least one action, so its thread never exits early)
    } else { a.slice_v = nullptr; a.slice_a = nullptr; }
    const dim3 grid(gx, gy, (unsigned)parts);
    const size_t smem = cash_diag_smem(D);
    const bool surv = m.recursion == SDPB_REC_SURVIVAL;
    cudaError_t e = cudaSuccess;
#define SDPB_DIAG_LAUNCH(SV, MN)                                                                              \
    {                                                                                                         \
        auto k = bi_cash_diag<SV, MN>;                                                                        \
        if (smem > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e == cudaSuccess) k<<<grid, kDiagCols, smem, stream>>>(dm, a);                                   \
    }
    if (surv) SDPB_DIAG_LAUNCH(true, false) else if (dm.is_min) SDPB_DIAG_LAUNCH(false, true) else SDPB_DIAG_LAUNCH(false, false)
#undef SDPB_DIAG_LAUNCH
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    if (parts > 1) {
        const unsigned mb = (unsigned)((n_local + 255) / 256);
        if (dm.is_min && !surv) merge_action_slices<true><<<mb, 256, 0, stream>>>(P.slice_v, P.slice_a, parts, n_local, Vt + lo, Qt + lo, lo, d_peers, n_peers, t);
        else merge_action_slices<false><<<mb, 256, 0, stream>>>(P.slice_v, P.slice_a, parts, n_local, Vt + lo, Qt + lo, lo, d_peers, n_peers, t);
        if (cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    }
    return SDPB_OK;
}

// ---------------------------------------------------------------------------------------------
// bi_cash_row — the cash-constraint family on ANY cash grid (fractional quantisers included), with the
// terms that do not depend on the cash level hoisted out of the thread.
//
// bi_generic evaluates the whole lambda per (state, action, demand): ~85 instructions per evaluation, and the
// lanes of a warp (consecutive cash levels of ONE inventory level) recompute identical revenue, holding cost,
// salvage and successor-row values.  Here a CTA is one inventory level x 128 cash levels; per action the CTA
// tabulates, one demand point per thread and with the reference's own double arithmetic
// (CashConstraint.java:103-121 via immediate<>'s expressions),
//     (1-rho)*price*min(y,d),  h*max(y-d,0),  salvage*max(y-d,0),  p,  p*gamma,  successor row offset,
// and a thread then only runs the cash-dependent tail of the lambda -- the deposit chain, the bankruptcy
// penalty, the clamp and the quantiser -- exactly as immediate<> / successor32<> write it.  Same operations in
// the same order on the same operands: bit-identical to bi_generic.
struct CashRowEntry {
    double rev1, hold, sal, p, pg;
    int row, pad;
};

template <bool SURVIVAL, bool IS_MIN>
__global__ void __launch_bounds__(128)
bi_cash_row(const __grid_constant__ DevModel M, const int t, const int D, const int pmf_off,
            const double* __restrict__ Vn, double* __restrict__ Vt, int* __restrict__ Qt,
            const long long lo, const long long hi, const long long row0, const int segs) {
    constexpr int KIND = SDPB_COST_CASH_DEPOSIT;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CashRowEntry* TB = reinterpret_cast<CashRowEntry*>(smem_raw);
    const int seg = (int)(blockIdx.x % segs);
    const long long ixl = row0 + blockIdx.x / segs;
    const int iw = min(seg * 128 + (int)threadIdx.x, M.nW - 1);
    const long long idx = ixl * M.nW + iw;
    const bool valid = seg * 128 + (int)threadIdx.x < M.nW && idx >= lo && idx < hi;
    const StateCtx S = decode_state<KIND>(M, t, idx);
    // the richest lane of the CTA has the longest action list: the cash bound of CashConstraint.java:96-99 grows with w
    // for a unit cost without its sign bit, which the host requires (cash_bound_grows_with_w)
    const StateCtx Stop = decode_state<KIND>(M, t, ixl * M.nW + min(seg * 128 + 127, M.nW - 1));
    const int nA_cta = Stop.nA;
    const double2* __restrict__ rec = M.pmf_rec + 2 * (size_t)pmf_off;

    double best = IS_MIN ? DBL_MAX : -DBL_MAX;
    int besti = kNoAction;
    for (int i = 0; i < nA_cta; i++) {
        const ActionCtx A = prep_action<KIND>(M, S, i);  // per lane: deposite depends on w
        __syncthreads();  // the previous action's table is no longer read
        for (int j = threadIdx.x; j < D; j += 128) {
            const double2 dp = __ldg(rec + 2 * j), gi = __ldg(rec + 2 * j + 1);
            const double d = dp.x;
            const double lvl = A.stock - d;                       // stock = x + a: the same for every lane
            const double revenue = S.price * jmin(A.stock, d);
            CashRowEntry e;
            e.rev1 = M.one_minus_rho * revenue;
            e.hold = M.h * jmax0(lvl);
            e.sal = S.last ? M.salvage * jmax0(lvl) : 0.0;
            e.p = dp.y;
            e.pg = gi.x;
            int il = A.iy - __double2loint(gi.y);
            if (S.lost) il = max(il, M.i_zero);
            il = min(il, M.nI - 1);
            il = max(il, 0);
            e.row = il * (int)S.strideX;
            e.pad = 0;
            TB[j] = e;
        }
        __syncthreads();
        if (!valid || i >= S.nA) continue;
        double acc = 0.0;
        for (int j = 0; j < D; j++) {
            const CashRowEntry e = TB[j];
            double inc = (((e.rev1 + A.deposite) - e.hold) - S.ovh) - A.initCash;  // CashConstraint.java:110
            inc += e.sal;
            const double endCash = A.initCash + inc;                               // CashConstraint.java:116-119
            if (endCash < 0.0) inc += M.pen * endCash;
            if (!SURVIVAL) acc += e.p * inc;                                       // CashRecursion.java:117
            if (Vn == nullptr) {  // period T without a boundary function
                if (SURVIVAL) {                                                    // RiskRecursion.java:80-84
                    const double finalCash = A.initCash + inc;
                    acc += e.p * (finalCash >= 0.0 ? 1.0 : 0.0);
                }
            } else {
                // successor32<> from the clamp on (CashConstraint.java:125-131)
                double nw = A.initCash + inc;
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
                int kw = k - (int)M.kmin;
                kw = max(min(kw, M.nW - 1), 0);
                double vn = __ldg(Vn + (e.row + kw));
                if (SURVIVAL && k < 0) vn = 0.0;                                   // RiskRecursion.java:87-95
                acc += e.pg * vn;                                                  // CashRecursion.java:120
            }
        }
        if (IS_MIN ? (acc < best) : (acc > best)) { best = acc; besti = i; }
    }
    if (valid) {
        Vt[idx] = best;
        Qt[idx] = besti == kNoAction ? -1 : besti;
    }
}

// ---------------------------------------------------------------------------------------------
// bi_cash_tail -- the row-shared kernel again, for the cash-constraint AND the overdraft lambdas
// (CashConstraint.java:95-133; CashOverdraft.java:72-118; CashOverdraftLimit.java:62-99; CashOverdraftTesting.java:78-120), with the per-lane tail cut to what the reference's
// arithmetic strictly needs.  ncu on bi_cash_row / bi_generic<OVERDRAFT> (profiles/r02_ncu_cash_row.md): 57 and 97
// warp instructions per evaluation, of which 21 and 20 on the fp64 pipe (each takes two dispatch slots); the rest is
// the clamp / round / convert / index sequence and reloads of model constants.  Here:
//   * the cash clamp moves behind the rounding: Math.round(x * q) is monotone, so
//     round(clamp(w', lo, hi) * q) == clamp(round(w' * q), round(lo * q), round(hi * q)) -- two integer min/max
//     instead of two fp64 compares and four selects (the host checks |w' * q| < 2^30 for every reachable w');
//   * the grid index needs no second clamp (the integer clamp already lands on the cash axis);
//   * `inc += salvage term` is skipped outside the last period (the term is +0.0 and inc is never -0.0: revenue
//     >= +0.0 for a non-negative price), the bankruptcy penalty when its rate is 0 (it would add -0.0);
//   * model constants live in registers, the demand loop is unrolled by two.
// Same operations on the same operands in the same order as immediate<> / successor32<> otherwise: bit-identical
// to bi_generic (tests: whole grid, both kinds, fractional and integer cash grids, gamma < 1, fuzz).
struct CashTailEntry {  // three 16-byte words: (rev, hold) (sal, p) (pg, row | pad)
    double rev, hold, sal, p, pg;
    int row, pad;
};
static_assert(sizeof(CashTailEntry) == 48, "three LDS.128 per entry");

// MODE: 0 = a period with a successor and no salvage term (t < T), 1 = period T without a successor, 2 = period T
// with a boundary table.  PEN: the bankruptcy penalty of CashConstraint.java:116-119 has a non-zero rate.
// DIV: the quantiser divides the rounded integer by q_div in long arithmetic (CashOverdraft.java:116), by multiply and
// shift (the host checks that every clamped integer is inside the exact range of the magic constant).
template <int KIND, int MODE, bool PEN, bool DIV>
__global__ void __launch_bounds__(128)
bi_cash_tail(const __grid_constant__ DevModel M, const int t, const int D, const int pmf_off,
             const double* __restrict__ Vn, double* __restrict__ Vt, int* __restrict__ Qt,
             const long long lo, const long long hi, const long long row0, const int segs, const int kk_lo_, const int kk_hi_) {
    constexpr bool LAST = MODE != 0, NEXT = MODE != 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CashTailEntry* TB = reinterpret_cast<CashTailEntry*>(smem_raw);
    const int seg = (int)(blockIdx.x % segs);
    const long long ixl = row0 + blockIdx.x / segs;
    const int iw = min(seg * 128 + (int)threadIdx.x, M.nW - 1);
    const long long idx = ixl * M.nW + iw;
    const bool valid = seg * 128 + (int)threadIdx.x < M.nW && idx >= lo && idx < hi;
    const StateCtx S = decode_state<KIND>(M, t, idx);
    const StateCtx Stop = decode_state<KIND>(M, t, ixl * M.nW + min(seg * 128 + 127, M.nW - 1));  // longest action list (bi_cash_row)
    const int nA_cta = Stop.nA;
    const double2* __restrict__ rec = M.pmf_rec + 2 * (size_t)pmf_off;
    // constants of the tail, in registers
    const double q_mul = M.q_mul, pen = M.pen, ovh = S.ovh;
    const int kk_lo = kk_lo_, kk_hi = kk_hi_;
    const unsigned q_magic_lo = (unsigned)M.q_magic;  // < 2^32 for q_div >= 2^15 is excluded by the plan: magic = ceil(2^47 / d)
    const unsigned long long q_magic = M.q_magic;
    const bool is_min = M.is_min != 0;
    (void)q_magic_lo;
    const unsigned tb_s = (unsigned)__cvta_generic_to_shared(TB);

    double best = is_min ? DBL_MAX : -DBL_MAX;
    int besti = kNoAction;
    for (int i = 0; i < nA_cta; i++) {
        const ActionCtx A = prep_action<KIND>(M, S, i);  // per lane: the deposit / interest terms depend on w
        __syncthreads();  // the previous action's table is no longer read
        for (int j = threadIdx.x; j < D; j += 128) {
            const double2 dp = __ldg(rec + 2 * j), gi = __ldg(rec + 2 * j + 1);
            const double d = dp.x;
            const double lvl = A.stock - d;                       // stock = x + a: the same for every lane
            const double revenue = S.price * jmin(A.stock, d);
            CashTailEntry e;
            e.rev = KIND == SDPB_COST_CASH_DEPOSIT ? M.one_minus_rho * revenue : revenue;
            e.hold = KIND != SDPB_COST_CASH_OVERDRAFT ? M.h * jmax0(lvl) : 0.0;
            e.sal = (LAST && KIND != SDPB_COST_CASH_OD_TESTING) ? M.salvage * jmax0(lvl) : 0.0;
            e.p = dp.y;
            e.pg = gi.x;
            int il = A.iy - __double2loint(gi.y);
            if (S.lost) il = max(il, M.i_zero);
            il = min(il, M.nI - 1);
            il = max(il, 0);
            e.row = il * (int)S.strideX - (int)M.kmin;  // + cash index k = flattened successor
            e.pad = 0;
            TB[j] = e;
        }
        __syncthreads();
        if (!valid || i >= S.nA) continue;
        const double initCash = A.initCash;
        double lane_term = KIND == SDPB_COST_CASH_DEPOSIT ? A.deposite : A.before_minus_interest;
        if (KIND == SDPB_COST_CASH_OD_LIMIT) lane_term = (S.w - A.fixedCost) - A.variableCost;  // CashOverdraftLimit.java:73
        const double r2 = M.r2, dr = M.dr, fixedCost = A.fixedCost, variableCost = A.variableCost;
        double acc = 0.0;
        unsigned ea = tb_s;
#pragma unroll 4
        for (int j = 0; j < D; j++, ea += (unsigned)sizeof(CashTailEntry)) {
            const double2 e0 = lds_double2(ea);          // (rev, hold)
            const double2 e1 = lds_double2(ea + 16u);    // (sal, p)
            const double2 e2 = lds_double2(ea + 32u);    // (pg, row in the low word)
            double inc, after_t = 0.0;
            if (KIND == SDPB_COST_CASH_DEPOSIT) {
                inc = (((e0.x + lane_term) - e0.y) - ovh) - initCash;           // CashConstraint.java:110
            } else if (KIND == SDPB_COST_CASH_OD_LIMIT) {                        // CashOverdraftLimit.java:70-86
                const double before = (lane_term - e0.y) - ovh;
                const double interest = r2 * jmax0(-before);
                const double deposite = dr * jmax0(before);
                const double bal = ((before - interest) + deposite) + e0.x;
                inc = bal - initCash;
            } else if (KIND == SDPB_COST_CASH_OD_TESTING) {                      // CashOverdraftTesting.java:85-99
                const double before = (((initCash + e0.x) - fixedCost) - variableCost) - e0.y;
                const double interest = r2 * jmax0(-before);
                after_t = before - interest;
                inc = after_t - initCash;
            } else {
                const double after = lane_term + e0.x;                           // CashOverdraft.java:99
                inc = after - initCash;
            }
            if (LAST && KIND != SDPB_COST_CASH_OD_TESTING) inc += e1.x;          // (+0.0 otherwise: see above)
            // end cash: w + c, except that CashOverdraftTesting.java:103-111 keeps the balance it computed
            double nw = KIND == SDPB_COST_CASH_OD_TESTING ? after_t : initCash + inc;
            if (PEN) {                                                           // CashConstraint.java:116-119
                const double inc2 = inc + pen * nw;
                const bool neg = nw < 0.0;
                inc = neg ? inc2 : inc;
                if (NEXT) nw = neg ? initCash + inc2 : nw;
            }
            acc += e1.y * inc;                                                   // CashRecursion.java:117
            if (NEXT) {
                int kk = jround32(nw * q_mul);                                   // Math.round(w' * q)
                kk = min(max(kk, kk_lo), kk_hi);                                 // the cash clamp, after the rounding
                int k = kk;
                if (DIV) {                                                       // Java long division, truncating toward zero
                    const unsigned a = (unsigned)(kk < 0 ? -kk : kk);
                    const int q = (int)(((unsigned long long)a * q_magic) >> 47);
                    k = kk < 0 ? -q : q;
                }
                acc += e2.x * __ldg(Vn + (__double2loint(e2.y) + k));           // CashRecursion.java:120
            }
        }
        if (is_min ? (acc < best) : (acc > best)) { best = acc; besti = i; }
    }
    if (valid) {
        Vt[idx] = best;
        Qt[idx] = besti == kNoAction ? -1 : besti;
    }
}

struct CashTailPlan { bool ok = false, div = false; int kk_lo = 0, kk_hi = 0; };

// The row kernels give every lane of a CTA the action count of its richest lane.  The cash-limited bound
// max(0, ((w - reserve) - reserve2) / v) grows with w for v > 0 and v = +0.0 (inf above the reserve, NaN on it), and
// falls for v < 0 and v = -0.0, where the poorer lanes would lose actions: such models go to the generic kernel.
inline bool cash_bound_grows_with_w(const sdpb_model& m) {
    if (!(m.flags & SDPB_F_CASH_LIMITED_ACTIONS)) return true;
    for (int t = 0; t < m.T; t++)
        if (std::signbit(m.vari_cost_t ? m.vari_cost_t[t] : m.vari_cost)) return false;
    return true;
}

// Both row-shared kinds, expectation recursion, no lead time, a rounding quantiser, 32-bit grid; every w' * q the
// kernel can form must stay below 2^30 in magnitude (jround32's low-word read and the integer clamp).
inline CashTailPlan plan_cash_tail(const sdpb_model& m, const DevModel& d, int D, const double* pmf_d, int n_pmf) {
    CashTailPlan P;
    if (!(m.cost_kind == SDPB_COST_CASH_DEPOSIT || m.cost_kind == SDPB_COST_CASH_OVERDRAFT ||
          m.cost_kind == SDPB_COST_CASH_OD_LIMIT || m.cost_kind == SDPB_COST_CASH_OD_TESTING)) return P;
    if (m.recursion != SDPB_REC_EXPECT || m.lead_time != 0 || d.small == 0 || m.quantiser == SDPB_Q_TRUNC) return P;
    if ((size_t)D * sizeof(CashTailEntry) > 96 * 1024 || !cash_bound_grows_with_w(m)) return P;
    if (m.cost_kind == SDPB_COST_CASH_DEPOSIT && !(1.0 - m.overhead_rate >= 0.0)) return P;
    double price = std::fabs(m.price), v = std::fabs(m.vari_cost), ovh = std::fabs(m.overhead), dmax = 0;
    for (int t = 0; t < m.T; t++) {
        const double pt = m.price_t ? m.price_t[t] : m.price;
        if (!(pt >= 0.0)) return P;  // revenue must never be -0.0 (see the kernel's header)
        price = std::max(price, std::fabs(pt));
        if (m.vari_cost_t) v = std::max(v, std::fabs(m.vari_cost_t[t]));
        if (m.overhead_t) ovh = std::max(ovh, std::fabs(m.overhead_t[t]));
    }
    for (int j = 0; j < n_pmf; j++) dmax = std::max(dmax, std::fabs(pmf_d[j]));
    const double stock = std::max(std::fabs(m.inv_min), std::fabs(m.inv_max)) + (double)m.max_order_idx * m.step;
    const double cash = std::max(std::fabs(m.cash_min), std::fabs(m.cash_max));
    const double rates = 1.0 + std::fabs(m.deposit_rate) + std::fabs(m.r0) + std::fabs(m.r2) + std::fabs(m.r3) + std::fabs(m.penalty_cost);
    // |w'| <= (cash + costs) * (1 + rates) + revenue + salvage/holding terms, generously
    const double bound = (cash + std::fabs(m.fixed_cost) + v * m.max_order_idx * m.step + ovh + std::fabs(m.od_limit) +
                          std::fabs(m.interest_free)) * rates * rates +
                         (price + std::fabs(m.salvage) + std::fabs(m.hold_cost)) * (stock + dmax) * rates;
    if (!(bound * std::fabs(m.q_mul) < 1073741824.0)) return P;
    auto hround = [](double x) { const double r = std::floor(x); return (long long)r + ((x - r) >= 0.5 ? 1 : 0); };
    P.kk_lo = (int)hround(m.cash_min * m.q_mul);
    P.kk_hi = (int)hround(m.cash_max * m.q_mul);
    P.div = m.quantiser == SDPB_Q_LONGDIV && d.q_idiv != 1;
    if (P.div) {  // the multiply-shift division is exact for |kk| < q_div * 2^16 with q_div < 2^15 (dev_model.cuh: jdiv32)
        const long long lim = d.q_idiv << 16;
        if (d.q_magic == 0 || std::llabs((long long)P.kk_lo) >= lim || std::llabs((long long)P.kk_hi) >= lim) return P;
    }
    P.ok = true;
    return P;
}

inline int launch_cash_tail(const CashTailPlan& P, const sdpb_model& m, const DevModel& dm, int t, int D, int pmf_off,
                            const double* Vn, double* Vt, int* Qt, long long lo, long long hi, cudaStream_t stream) {
    if (hi <= lo) return SDPB_OK;
    const int segs = (dm.nW + 127) / 128;
    const long long row0 = lo / dm.nW, row1 = (hi - 1) / dm.nW;
    const unsigned blocks = (unsigned)((row1 - row0 + 1) * segs);
    const size_t smem = (size_t)D * sizeof(CashTailEntry);
    cudaError_t e = cudaSuccess;
#define SDPB_TAIL_LAUNCH(KD, MD, PN, DV)                                                                \
    {                                                                                                   \
        auto k = bi_cash_tail<KD, MD, PN, DV>;                                                          \
        if (smem > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e == cudaSuccess) k<<<blocks, 128, smem, stream>>>(dm, t, D, pmf_off, Vn, Vt, Qt, lo, hi, row0, segs, P.kk_lo, P.kk_hi); \
    }
#define SDPB_TAIL_MODE(KD, PN, DV)                                                                      \
    { if (mode == 0) SDPB_TAIL_LAUNCH(KD, 0, PN, DV) else if (mode == 1) SDPB_TAIL_LAUNCH(KD, 1, PN, DV) else SDPB_TAIL_LAUNCH(KD, 2, PN, DV) }
    const int mode = t < m.T ? 0 : (Vn == nullptr ? 1 : 2);
    if (m.cost_kind == SDPB_COST_CASH_DEPOSIT) {
        const bool pn = m.penalty_cost != 0.0;
        if (pn) { if (P.div) SDPB_TAIL_MODE(SDPB_COST_CASH_DEPOSIT, true, true) else SDPB_TAIL_MODE(SDPB_COST_CASH_DEPOSIT, true, false) }
        else    { if (P.div) SDPB_TAIL_MODE(SDPB_COST_CASH_DEPOSIT, false, true) else SDPB_TAIL_MODE(SDPB_COST_CASH_DEPOSIT, false, false) }
    } else if (m.cost_kind == SDPB_COST_CASH_OD_LIMIT) {
        if (P.div) SDPB_TAIL_MODE(SDPB_COST_CASH_OD_LIMIT, false, true) else SDPB_TAIL_MODE(SDPB_COST_CASH_OD_LIMIT, false, false)
    } else if (m.cost_kind == SDPB_COST_CASH_OD_TESTING) {
        if (P.div) SDPB_TAIL_MODE(SDPB_COST_CASH_OD_TESTING, false, true) else SDPB_TAIL_MODE(SDPB_COST_CASH_OD_TESTING, false, false)
    } else {
        if (P.div) SDPB_TAIL_MODE(SDPB_COST_CASH_OVERDRAFT, false, true) else SDPB_TAIL_MODE(SDPB_COST_CASH_OVERDRAFT, false, false)
    }
#undef SDPB_TAIL_MODE
#undef SDPB_TAIL_LAUNCH
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    return SDPB_OK;
}

// CASH_DEPOSIT kind without lead time on a grid whose indices fit 32 bits (DevModel::small), with a cash bound that
// grows with w.
inline bool cash_row_ok(const sdpb_model& m, const DevModel& d, int D) {
    return m.cost_kind == SDPB_COST_CASH_DEPOSIT && m.lead_time == 0 && d.small != 0 &&
           (size_t)D * sizeof(CashRowEntry) <= 96 * 1024 && cash_bound_grows_with_w(m);
}

inline int launch_cash_row(const sdpb_model& m, const DevModel& dm, int t, int D, int pmf_off, const double* Vn,
                           double* Vt, int* Qt, long long lo, long long hi, cudaStream_t stream) {
    if (hi <= lo) return SDPB_OK;
    const int segs = (dm.nW + 127) / 128;
    const long long row0 = lo / dm.nW, row1 = (hi - 1) / dm.nW;
    const unsigned blocks = (unsigned)((row1 - row0 + 1) * segs);
    const size_t smem = (size_t)D * sizeof(CashRowEntry);
    const bool surv = m.recursion == SDPB_REC_SURVIVAL;
    cudaError_t e = cudaSuccess;
#define SDPB_ROW_LAUNCH(SV, MN)                                                                         \
    {                                                                                                   \
        auto k = bi_cash_row<SV, MN>;                                                                   \
        if (smem > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e == cudaSuccess) k<<<blocks, 128, smem, stream>>>(dm, t, D, pmf_off, Vn, Vt, Qt, lo, hi, row0, segs); \
    }
    if (surv) SDPB_ROW_LAUNCH(true, false) else if (dm.is_min) SDPB_ROW_LAUNCH(false, true) else SDPB_ROW_LAUNCH(false, false)
#undef SDPB_ROW_LAUNCH
    if (e != cudaSuccess || cudaGetLastError() != cudaSuccess) return SDPB_ERR_CUDA;
    return SDPB_OK;
}

}  // namespace sdpb
