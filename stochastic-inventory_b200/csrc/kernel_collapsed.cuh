// kernel_collapsed.cuh — OPT-IN collapsed solve of the 1-D inventory family (SDPB_KERNEL_COLLAPSED, request only).
//
// NOT bit-identical to the reference, and never chosen by SDPB_KERNEL_AUTO.  The reference evaluates, per (x, a),
//     Q(x, a) = sum_j [ p_j * ((fixed + v*a) + L(x + a - d_j))  +  (p_j*gamma) * V_{t+1}(x + a - d_j) ]
// (Recursion.java:129-161 with the lambdas of CLSPTesting.java:78-106).  Everything but the ordering cost depends on
// (x, a) only through the order-up-to level y = x + a, so in exact arithmetic
//     Q(x, a) = (fixed + v*a) * sum_j p_j + G(y),   G(y) = sum_j p_j * L(y - d_j) + sum_j (p_j*gamma) * V_{t+1}(y - d_j),
// and with sum_j p_j = 1 the solve is one pass of D operations per LEVEL plus one pass of A operations per state
// instead of A * D per state: C5 at 1e7 states goes from 305 ms to a few ms.  In floating point the two differ by the
// rounding of a 200-term sum and by 1 - sum_j p_j (~1e-16 for the pmf tables of getpmf.py): values agree to ~1e-13
// relative -- inside the 1e-9 the task statement allows, outside the bit-exactness every other kernel of the library
// keeps -- and the argmin can move between actions whose values differ by less than that.  Callers who want the
// reference's tables bit for bit do not set this kernel; bench.py reports it as its own line and never in evals/s.
// stats.evals keeps counting the reference's evaluations, stats.evals_executed what ran.
#pragma once
#include <cuda_runtime.h>

#include "dev_model.cuh"

namespace sdpb {

// Level costs L(il) = h*max(lvl,0) + pi*max(-lvl,0) for il in [il0, il0 + n): model constants only, tabulated once per handle
__global__ void __launch_bounds__(256)
collapsed_level_costs(const __grid_constant__ DevModel M, const long long il0, const long long n, double* __restrict__ Lc) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double lvl = M.inv_min + (double)(il0 + i) * M.step;
    Lc[i] = M.h * fmax(lvl, 0.0) + M.pen * fmax(-lvl, 0.0);
}

// G over the level indices y = ix + ia in [0, nY), nY = nI + max_order_idx (level value = inv_min + y*step).
// Lanes hold consecutive y: for each demand point the level cost and the successor value are coalesced lines.
template <bool LAST>
__global__ void __launch_bounds__(256)
collapsed_levels(const __grid_constant__ DevModel M, const int D, const int pmf_off, const double* __restrict__ Vn,
                 const double* __restrict__ Lc, const long long il0, double* __restrict__ G, const int nY) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2* PJ = reinterpret_cast<double2*>(smem_raw);           // (p_j, p_j*gamma)
    int* DJ = reinterpret_cast<int*>(smem_raw + (size_t)D * 16);  // d_j / step
    for (int j = threadIdx.x; j < D; j += blockDim.x) {
        PJ[j] = make_double2(M.pmf_p[pmf_off + j], M.pmf_pg[pmf_off + j]);
        DJ[j] = M.pmf_di[pmf_off + j];
    }
    __syncthreads();
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= nY) return;
    const int lo_clamp = (M.flags & SDPB_F_LOST_SALES) ? max(M.i_zero, 0) : 0;  // (levels below zero lift to the zero row)
    const int hi_clamp = M.nI - 1;
    const double* __restrict__ lc = Lc - il0;
    double acc = 0.0;
#pragma unroll 4
    for (int j = 0; j < D; j++) {
        const int il = y - DJ[j];
        const double2 pj = PJ[j];
        acc += pj.x * __ldg(lc + il);
        if (!LAST) {
            const int is = max(min(il, hi_clamp), lo_clamp);  // upper clamp first (CLSPTesting.java:91-92)
            acc += pj.y * __ldg(Vn + is);
        }
    }
    G[y] = acc;
}

// V_t(x) = opt_a (fixed 1[a>0] + v*a) + G(x + a), first optimum wins (Recursion.java:146-157).  The ordering costs are
// tabulated once per CTA; lanes hold consecutive states, so G(x + a) is one coalesced line per warp and action.
template <bool IS_MIN>
__global__ void __launch_bounds__(256)
collapsed_actions(const __grid_constant__ DevModel M, const int t, const double* __restrict__ G,
                  double* __restrict__ Vt, int* __restrict__ Qt, const long long S) {
    extern __shared__ double FV[];  // [max_order_idx + 1]
    const double v = M.v_t[t - 1];
    for (int a = threadIdx.x; a <= M.max_order_idx; a += blockDim.x) {
        const double av = (double)a * M.step;
        FV[a] = (av > 0.0 ? M.K : 0.0) + v * av;
    }
    __syncthreads();
    const long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= S) return;
    const double* __restrict__ g = G + x;
    double best = IS_MIN ? DBL_MAX : -DBL_MAX;
    int arg = -1;
#pragma unroll 4
    for (int a = 0; a <= M.max_order_idx; a++) {
        const double q = FV[a] + __ldg(g + a);
        if (IS_MIN ? (q < best) : (q > best)) { best = q; arg = a; }
    }
    Vt[x] = best;
    Qt[x] = arg;
}

inline bool collapsed_ok(const sdpb_model& m) {
    return m.cost_kind == SDPB_COST_BACKORDER && m.lead_time == 0 && (m.flags & SDPB_F_CLAMP_INV) &&
           !(m.flags & SDPB_F_GY_MODE) && !(m.flags & SDPB_F_NO_ORDER_LAST) && m.max_order_idx < 6000;
}

inline int launch_collapsed(const DevModel& dm, int t, int D, int pmf_off, const double* Vn, const double* Lc,
                            long long il0, double* G, double* Vt, int* Qt, cudaStream_t stream) {
    const int nY = dm.nI + dm.max_order_idx;
    const unsigned gb = (unsigned)((nY + 255) / 256), sb = (unsigned)((dm.S + 255) / 256);
    // both below 48 KB: sdpb_create refuses max_order_idx >= 6000 and demand rows longer than 2000 for this kernel
    const size_t smem_l = (size_t)D * 20 + 16;
    const size_t smem = (size_t)(dm.max_order_idx + 1) * sizeof(double);
    if (Vn) collapsed_levels<false><<<gb, 256, smem_l, stream>>>(dm, D, pmf_off, Vn, Lc, il0, G, nY);
    else collapsed_levels<true><<<gb, 256, smem_l, stream>>>(dm, D, pmf_off, Vn, Lc, il0, G, nY);
    if (dm.is_min) collapsed_actions<true><<<sb, 256, smem, stream>>>(dm, t, G, Vt, Qt, dm.S);
    else collapsed_actions<false><<<sb, 256, smem, stream>>>(dm, t, G, Vt, Qt, dm.S);
    return cudaGetLastError() == cudaSuccess ? SDPB_OK : SDPB_ERR_CUDA;
}

}  // namespace sdpb
