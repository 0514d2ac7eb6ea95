// sdpb200.cu — the C-ABI of libsdpb200.so (include/sdpb200.h): descriptor validation, device
// tables, one kernel launch per period, result extraction.  No CPU solve path exists here: if the
// device is missing every entry point fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include <unistd.h>

#include "../../include/sdpb200.h"
#include "dev_model.cuh"
#include "kernel_generic.cuh"
#include "kernel_tiled.cuh"
#include "kernel_lead.cuh"
#include "kernel_cash.cuh"
#include "kernel_two_product.cuh"
#include "kernel_staff.cuh"
#include "kernel_collapsed.cuh"
#include "kernel_fused.cuh"
#include "microbench.cuh"

using namespace sdpb;

namespace {

thread_local std::string g_create_error;

inline long long h_jround(double x) {  // Math.round(double)
    double r = std::floor(x);
    return (long long)r + ((x - r) >= 0.5 ? 1 : 0);
}
inline bool is_int(double x) { return std::isfinite(x) && x == std::floor(x) && std::fabs(x) < 1e15; }

#define CU(call)                                                                        \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) {                                                        \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                \
            return SDPB_ERR_CUDA;                                                       \
        }                                                                               \
    } while (0)

template <class T>
int upload(sdpb_handle* h, const std::vector<T>& v, T** out);

}  // namespace

// ---- multi-GPU: the other shards' tables, mapped into this process ------------------------------------------
// What one shard tells the others (sdpb_peer_export): plain bytes, SDPB_PEER_BLOB_BYTES of them.
struct PeerInfo {
    uint32_t magic, version;
    int32_t rank, world, device, T;
    int64_t pid;
    uint64_t base;             // slab address in the exporting process (used when importer and exporter share a process)
    int64_t n_states, lo, hi;  // grid size, owned block
    int64_t rlo, rhi;          // rows its kernels read (sdpb_shard_reads)
    int64_t vlo, vhi;          // window it holds
    uint64_t v_off0, v_stride; // address of V_t[i] = base + v_off0 + (t-1) * v_stride + (i - vlo) * 8
    uint64_t flags_off;        // unsigned[64]: flags[r] = number of exchanges rank r has completed into this shard
    uint64_t model_hash;
    uint64_t handle;           // the exporting sdpb_handle* (meaningful in the exporting process only)
    char pci[24];              // PCI bus id of the exporter's GPU: two PROCESSES must not share a GPU (see sdpb_peer_attach)
    cudaIpcMemHandle_t ipc;
};
static_assert(sizeof(PeerInfo) <= SDPB_PEER_BLOB_BYTES, "peer blob too small");
constexpr uint32_t kPeerMagic = 0x53445042u;  // "SDPB"
constexpr int kMaxPeers = 64;
constexpr size_t kSlabHeader = 1024;          // flags[64], error word, padding

struct PeerSend { int rank; long long a, b; };  // rows [a, b) of my block that peer `rank` reads
struct PeerLink {
    bool attached = false;
    std::vector<PeerInfo> info;        // [world]
    std::vector<char*> mapped;         // [world] peers' slabs in this address space (own slab for own rank)
    std::vector<char> ipc_opened;      // [world] mapped with cudaIpcOpenMemHandle (must be closed)
    std::vector<PeerSend> sends;
    std::vector<int> recv_from;
    void* d_peers = nullptr;           // device array of DevPeer, one per entry of `sends` (kernels that push themselves)
    unsigned** d_targets = nullptr;    // device array: address of flags[my rank] in every peer I send to
    int* d_from = nullptr;             // device array: ranks I wait for
    unsigned epoch = 0;                // exchanges completed so far (identical on every shard)
    long long bytes_out = 0, bytes_in = 0;
    // Hand-over of the pushed rows.  Shards in different processes (one per GPU): a flag word in the receiver's memory,
    // stored after the copies and spun on by a one-CTA kernel of the receiver.  Shards of ONE process (sdpb_group_*):
    // a CUDA event recorded after the copies, which the receivers' streams wait on -- no kernel ever waits for another
    // kernel, so shards may share a GPU (kernels that spin on each other are not guaranteed to run at the same time).
    bool by_events = false;
    cudaEvent_t ev_pushed = nullptr;
    std::vector<sdpb_handle*> peer_handles;  // [world], by_events only
};

struct sdpb_handle {
    sdpb_model m{};
    DevModel dm{};
    sdpb_options opt{};
    std::vector<int> pmf_len, pmf_off;
    std::vector<double> pmf_d, pmf_p;
    std::vector<int> pmf_di;  // demand values in units of step
    std::vector<double> pmf_d2;
    std::vector<int> apmf_len;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int ndim = 1;
    long long S = 0, Spad = 0, lo = 0, hi = 0;
    std::vector<double*> dV;  // [T] each Spad doubles (full grid: period t-1 reads all of period t)
    std::vector<int*> dQ;     // [T] each Spad int32 action indices (-1 = none)
    std::vector<unsigned char*> dMask;  // [T] reachability, one byte per state
    std::vector<char> solved;
    mutable std::vector<double> evals_cache;
    std::vector<void*> dev_allocs;
    bool reached = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    sdpb_stats stats{};
    TiledPlan tiled{};
    CashPlan cash{};
    FusedPlan fused{};
    int sm_count = 0;
    int solve_count = 0;
    cudaGraphExec_t graph_exec = nullptr;  // the T launches of one solve, captured on the second solve
    bool graph_failed = false;
    sdpb_stats graph_stats{};
    bool dedup = false;        // lead-time models: fold (x, preQ) -> x + preQ
    long long vS = 0;          // virtual states per period
    double* dHv = nullptr;     // [vS] virtual value table of the period being solved
    int* dHa = nullptr;        // [vS] virtual policy table
    double* dVT = nullptr;     // V_{t+1} with the two pipeline axes transposed (bi_lead_q2); indexed like dV
    double* dTerm = nullptr;   // terminal boundary table V_{T+1} (sdpb_model.terminal_value); indexed like dV
    // What is held in device memory.  dV[t][i] is valid for vlo <= i < vhi (the whole grid when unsharded, else
    // the rows this shard's kernels can read plus a guard margin) and dQ[t][i] for lo <= i < hi: the pointers are
    // biased so that kernels keep indexing with absolute flattened indices.
    long long vlo = 0, vhi = 0;
    size_t device_bytes = 0;
    char* slab = nullptr;      // sharded handles: ONE cudaMalloc allocation (CUDA IPC cannot export pool memory)
    size_t slab_bytes = 0;
    size_t v_off0 = 0, v_stride = 0;  // byte offset of element vlo of V_1 inside the slab; bytes between periods
    unsigned long long* dCounters = nullptr;  // [4] dense-grid artefacts seen by sdpb_reach
    double reach_cnt[3] = {0, 0, 0};
    PeerLink peer;
    std::vector<sdpb_kernel_choice> period_kernel;  // [T] choose_period_kernel
    bool push_fused = false;   // the period's kernel already stored the peers' rows into their tables (bi_lead_q2)
    double* q2_slice_v = nullptr;  // bi_lead_q2m with action slices over separate CTAs: per slice and state the slice's optimum
    int* q2_slice_a = nullptr;
    size_t q2_slice_cap = 0;
    double* dG = nullptr;          // SDPB_KERNEL_COLLAPSED: G over the nI + max_order order-up-to levels
    double* dLc = nullptr;         // ... and the level costs over [lc_il0, lc_il0 + n)
    long long lc_il0 = 0;
    std::vector<cudaEvent_t> prof_ev;  // profile = 1: 4 events per period
    std::vector<double> prof_ms;       // [3 * T] of the last sharded solve
    std::string err;
};

namespace {

// Device memory comes from a stream-ordered pool PRIVATE to this library (one per device) whose release
// threshold is lifted, so a create/solve/destroy cycle reuses the previous cycle's memory instead of paying
// cudaMalloc/cudaFree (cudaFree of the C5 tables alone cost 1.1 s per cycle).  The process-wide default pool
// is left alone: a JVM host's other libraries keep their allocator behaviour.  sdpb_trim_pool gives the cached
// memory back.
std::mutex g_pool_mu;
cudaMemPool_t g_pools[64] = {};

cudaMemPool_t library_pool(int dev) {
    if (dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (!g_pools[dev]) {
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        cudaMemPool_t pool = nullptr;
        if (cudaMemPoolCreate(&pool, &props) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        g_pools[dev] = pool;
    }
    return g_pools[dev];
}

// Sharded handles keep their tables in ONE plain cudaMalloc allocation (CUDA IPC cannot export pool memory).  cudaMalloc /
// cudaFree of a gigabyte and cudaIpcOpenMemHandle / cudaIpcCloseMemHandle cost 50-170 ms per create/destroy cycle, so a
// destroyed handle's slab is parked here and the next sharded handle of the device that fits reuses it; a peer that has
// mapped it before finds the mapping (keyed by the IPC handle's bytes) still open.  sdpb_trim_pool releases everything.
struct Slab { char* p; size_t bytes; };
std::vector<Slab> g_slabs[64];
struct IpcMapping { cudaIpcMemHandle_t handle; int device; char* p; };
std::vector<IpcMapping> g_ipc_maps;
constexpr size_t kMaxParkedSlabs = 4;

char* slab_acquire(int dev, size_t bytes, size_t* got) {
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        auto& v = g_slabs[dev];
        size_t best = v.size();
        for (size_t i = 0; i < v.size(); i++)
            if (v[i].bytes >= bytes && v[i].bytes <= bytes + bytes / 4 + (1u << 20) && (best == v.size() || v[i].bytes < v[best].bytes))
                best = i;
        if (best != v.size()) {
            char* p = v[best].p;
            *got = v[best].bytes;
            v.erase(v.begin() + (long)best);
            return p;
        }
    }
    char* p = nullptr;
    if (cudaMalloc((void**)&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    *got = bytes;
    return p;
}

void slab_release(int dev, char* p, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    auto& v = g_slabs[dev];
    if (v.size() >= kMaxParkedSlabs) {  // keep the most recent ones
        cudaFree(v.front().p);
        v.erase(v.begin());
    }
    v.push_back({p, bytes});
}

// A peer process's slab in this address space (for the CUDA device current at the call).
cudaError_t ipc_map(const cudaIpcMemHandle_t& hd, int device, char** out) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    for (const IpcMapping& m : g_ipc_maps)
        if (m.device == device && std::memcmp(&m.handle, &hd, sizeof hd) == 0) { *out = m.p; return cudaSuccess; }
    void* p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return e;
    g_ipc_maps.push_back({hd, device, (char*)p});
    *out = (char*)p;
    return cudaSuccess;
}

cudaError_t pool_alloc(sdpb_handle* h, void** p, size_t bytes) {
    cudaMemPool_t pool = library_pool(h->device);
    if (pool) return cudaMallocFromPoolAsync(p, std::max<size_t>(bytes, 16), pool, h->stream);
    return cudaMallocAsync(p, std::max<size_t>(bytes, 16), h->stream);
}

// long-lived allocation owned by the handle
cudaError_t dev_alloc(sdpb_handle* h, void** p, size_t bytes) {
    cudaError_t e = pool_alloc(h, p, bytes);
    if (e == cudaSuccess) { h->dev_allocs.push_back(*p); h->device_bytes += std::max<size_t>(bytes, 16); }
    return e;
}

template <class T>
int upload(sdpb_handle* h, const std::vector<T>& v, T** out) {
    void* p = nullptr;
    CU(dev_alloc(h, &p, v.size() * sizeof(T)));
    if (!v.empty()) CU(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    *out = (T*)p;
    return SDPB_OK;
}

int fail_create(sdpb_handle* h, int code, const std::string& msg) {
    g_create_error = msg;
    if (h) sdpb_destroy(h);
    return code;
}

bool has_cash(const sdpb_model& m) { return m.cost_kind != SDPB_COST_BACKORDER && m.cost_kind != SDPB_COST_STAFF; }
bool staff_kind(const sdpb_model& m) { return m.cost_kind == SDPB_COST_STAFF; }
bool two_product(const sdpb_model& m) { return m.cost_kind == SDPB_COST_CASH_TWO_PRODUCT; }

double cash_of_k(const sdpb_handle* h, long long k) {
    const sdpb_model& m = h->m;
    if (m.cost_kind == SDPB_COST_CASH_XR) return (double)k;
    return m.quantiser == SDPB_Q_DIV ? (double)k / m.q_div : (double)k;
}
double quantise(const sdpb_model& m, double w) {
    if (m.quantiser == SDPB_Q_TRUNC) return (double)(int)w;  // grid bounds: truncation only
    long long kk = h_jround(w * m.q_mul);
    if (m.quantiser == SDPB_Q_DIV) return (double)kk / m.q_div;
    return (double)(kk / (long long)m.q_div);
}
long long cash_k_of(const sdpb_model& m, double wq) {
    if (m.cost_kind == SDPB_COST_CASH_XR) return h_jround(wq);
    return m.quantiser == SDPB_Q_DIV ? h_jround(wq * m.q_div) : (long long)wq;
}

// API-order state -> flattened index, or -1 when it is not a grid point.
long long index_of_state(const sdpb_handle* h, const double* st) {
    const sdpb_model& m = h->m;
    const DevModel& d = h->dm;
    int k = 0;
    double x = st[k++];
    double fi = (x - m.inv_min) / m.step;
    if (!is_int(fi) || fi < 0 || fi >= d.nI) return -1;
    long long idx = (long long)fi;
    if (two_product(m)) {
        double f2 = (st[k++] - m.inv_min) / m.step;
        if (!is_int(f2) || f2 < 0 || f2 >= d.nI) return -1;
        idx = idx * d.nI + (long long)f2;
    }
    long long iw = 0;
    if (has_cash(m)) {
        double w = st[k++];
        long long kk = cash_k_of(m, w);
        if (cash_of_k(h, kk) != w) return -1;
        iw = kk - d.kmin;
        if (iw < 0 || iw >= d.nW) return -1;
    }
    for (int l = 0; l < m.lead_time; l++) {
        double q = st[k++];
        double fq = q / m.step;
        if (!is_int(fq) || fq < 0 || fq >= d.nQ) return -1;
        idx = idx * d.nQ + (long long)fq;
    }
    if (has_cash(m)) idx = idx * d.nW + iw;
    return idx;
}

void state_of_index(const sdpb_handle* h, long long idx, double* st, double* x_out) {
    const sdpb_model& m = h->m;
    const DevModel& d = h->dm;
    double w = 0, q1 = 0, q2 = 0;
    if (has_cash(m)) { w = cash_of_k(h, d.kmin + idx % d.nW); idx /= d.nW; }
    if (m.lead_time >= 2) { q2 = (double)(idx % d.nQ) * m.step; idx /= d.nQ; }
    if (m.lead_time >= 1) { q1 = (double)(idx % d.nQ) * m.step; idx /= d.nQ; }
    double x2 = 0;
    if (two_product(m)) { x2 = m.inv_min + (double)(idx % d.nI) * m.step; idx /= d.nI; }
    double x = m.inv_min + (double)idx * m.step;
    if (x_out) *x_out = x;
    if (st) {
        int k = 0;
        st[k++] = x;
        if (two_product(m)) st[k++] = x2;
        if (has_cash(m)) st[k++] = w;
        if (m.lead_time >= 1) st[k++] = q1;
        if (m.lead_time >= 2) st[k++] = q2;
    }
}

inline double q_of_index(const sdpb_handle* h, long long idx, int qi) {
    if (qi < 0) return 0.0;  // bestOrderQty stays 0 when nothing beat the initial value
    if (two_product(h->m)) return (double)qi;  // pair index Q1*(max_order_idx+1) + Q2
    if (h->m.cost_kind == SDPB_COST_CASH_XR) {
        double x;
        state_of_index(h, idx, nullptr, &x);
        return x + (double)qi * h->m.step;
    }
    return (double)qi * h->m.step;
}

// |A_t(s)| summed over the shard, times D_t (host arithmetic; mirrors decode_state()).
double count_evals_period_uncached(const sdpb_handle* h, int t);

// The shard never changes, so the (host-side) count is computed once per period.
double count_evals_period(const sdpb_handle* h, int t) {
    if (h->evals_cache.size() != (size_t)h->m.T) h->evals_cache.assign(h->m.T, -1.0);
    double& c = h->evals_cache[t - 1];
    if (c < 0) c = count_evals_period_uncached(h, t);
    return c;
}

double count_evals_period_uncached(const sdpb_handle* h, int t) {
    const sdpb_model& m = h->m;
    const DevModel& d = h->dm;
    const double D = h->pmf_len[t - 1];
    if (staff_kind(m)) {
        // sum over the shard's states and actions of the length of the pmf row they use
        double total = 0;
        const int* len = h->apmf_len.data() + (size_t)(t - 1) * d.nI;
        for (long long ix = h->lo; ix < h->hi; ix++)
            for (int i = 0; i <= m.max_order_idx; i++) total += len[std::min<long long>(ix + i, d.nI - 1)];
        return total;
    }
    if (two_product(m)) {
        // affordable pairs depend on the cash level only (MultiItemCash.java:73)
        const double v1 = m.vari_cost_t ? m.vari_cost_t[t - 1] : m.vari_cost;
        const int Q = m.max_order_idx + 1;
        double total = 0;
        for (int iw = 0; iw < d.nW; iw++) {
            const double w = (double)(d.kmin + iw);
            long long cnt = 0;
            for (int i = 0; i < Q; i++)
                for (int j = 0; j < Q; j++) cnt += (v1 * i + m.vari_cost2 * j < w + 0.1);
            // states of the shard [lo, hi) whose cash index is iw
            const long long n_iw = (h->hi - iw + d.nW - 1) / d.nW - (h->lo - iw + d.nW - 1) / d.nW;
            total += (double)cnt * (double)n_iw;
        }
        return total * D;
    }
    const long long n = h->hi - h->lo;
    const bool limited = (m.flags & SDPB_F_CASH_LIMITED_ACTIONS) || m.cost_kind == SDPB_COST_CASH_XR;
    if ((m.flags & SDPB_F_NO_ORDER_LAST) && t == m.T && m.cost_kind != SDPB_COST_CASH_XR) return (double)n * D;
    if (!limited) return (double)n * (m.max_order_idx + 1) * D;
    const double v = m.vari_cost_t ? m.vari_cost_t[t - 1] : m.vari_cost;
    const double res = m.reserve_t ? m.reserve_t[t - 1] : 0.0;
    double total = 0;
    // the action count depends on (x, w) only; walk the shard
    for (long long idx = h->lo; idx < h->hi; idx++) {
        long long r = idx;
        double w = cash_of_k(h, d.kmin + r % d.nW);
        r /= d.nW;
        for (int l = 0; l < m.lead_time; l++) r /= d.nQ;
        double x = m.inv_min + (double)r * m.step;
        int nA;
        if (m.cost_kind == SDPB_COST_CASH_XR) {
            double rv = w / v;
            double maxY = rv < x ? x : rv;
            nA = std::min((int)(maxY - x) + 1, m.max_order_idx + 1);
        } else {
            nA = (int)std::min((double)m.max_order_idx, std::max(0.0, ((w - res) - m.reserve2) / v)) + 1;
        }
        total += nA;
    }
    return total * D;
}

// Launch the general kernel over index range [lo, hi) of the real grid, or (DEDUP) of the virtual grid.
template <int KIND, bool SURV, bool IS_MIN, int G, bool DEDUP>
void launch_generic(sdpb_handle* h, int t, const double* Vn, double* Vt, int* Qt, long long lo, long long hi) {
    const long long n = hi - lo;
    if (n <= 0) return;
    const int per_block = 256 / G;
    const long long blocks = (n + per_block - 1) / per_block;
    bi_generic<KIND, SURV, IS_MIN, G, DEDUP><<<(unsigned)blocks, 256, 0, h->stream>>>(
        h->dm, t, h->pmf_len[t - 1], h->pmf_off[t - 1], Vn, Vt, Qt, lo, hi);
}

// The general kernel for every cost kind.  Only kinds with a lead time (backorder, deposit, overdraft) are ever folded.
template <bool DEDUP>
int dispatch_generic_d(sdpb_handle* h, int t, const double* Vn, double* Vt, int* Qt, long long lo, long long hi) {
    const sdpb_model& m = h->m;
    const bool surv = m.recursion == SDPB_REC_SURVIVAL;
    const bool mn = h->dm.is_min != 0;
    switch (m.cost_kind) {
    case SDPB_COST_BACKORDER:
        if (mn) launch_generic<SDPB_COST_BACKORDER, false, true, 32, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        else launch_generic<SDPB_COST_BACKORDER, false, false, 32, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        break;
    case SDPB_COST_CASH_DEPOSIT:
        if (surv) launch_generic<SDPB_COST_CASH_DEPOSIT, true, false, 1, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        else if (mn) launch_generic<SDPB_COST_CASH_DEPOSIT, false, true, 1, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        else launch_generic<SDPB_COST_CASH_DEPOSIT, false, false, 1, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        break;
    case SDPB_COST_CASH_OVERDRAFT:
        if (surv) launch_generic<SDPB_COST_CASH_OVERDRAFT, true, false, 1, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        else if (mn) launch_generic<SDPB_COST_CASH_OVERDRAFT, false, true, 1, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        else launch_generic<SDPB_COST_CASH_OVERDRAFT, false, false, 1, DEDUP>(h, t, Vn, Vt, Qt, lo, hi);
        break;
    case SDPB_COST_STAFF: {
        const long long nst = hi - lo;
        const bool last = Vn == nullptr;
        auto k = mn ? (last ? bi_staff<true, true> : bi_staff<true, false>) : (last ? bi_staff<false, true> : bi_staff<false, false>);
        if (nst > 0) k<<<(unsigned)((nst + 7) / 8), 256, 0, h->stream>>>(h->dm, t, Vn, Vt, Qt, lo, hi);
        break;
    }
    case SDPB_COST_CASH_TWO_PRODUCT: {
        const long long nst = hi - lo;
        const bool term_T = t == h->m.T && Vn != nullptr;  // boundary table: the kernel folds LAST and 'no continuation'
        auto k = term_T ? bi_two_product<true, true> : t == h->m.T ? bi_two_product<true, false> : bi_two_product<false, true>;
        if (nst > 0) k<<<(unsigned)((nst + 127) / 128), 128, 0, h->stream>>>(h->dm, t, h->pmf_len[t - 1], h->pmf_off[t - 1], Vn, Vt, Qt, lo, hi);
        break;
    }
#define SDPB_PLAIN_KIND(K)                                                                    \
    case K:                                                                                   \
        if (mn) launch_generic<K, false, true, 1, false>(h, t, Vn, Vt, Qt, lo, hi);           \
        else launch_generic<K, false, false, 1, false>(h, t, Vn, Vt, Qt, lo, hi);             \
        break;
    SDPB_PLAIN_KIND(SDPB_COST_CASH_XR)
    SDPB_PLAIN_KIND(SDPB_COST_CASH_OD_LIMIT)
    SDPB_PLAIN_KIND(SDPB_COST_CASH_OD_TESTING)
    SDPB_PLAIN_KIND(SDPB_COST_CASH_LOAN)
#undef SDPB_PLAIN_KIND
    default:
        h->err = "bad cost_kind";
        return SDPB_ERR_ARG;
    }
    return SDPB_OK;
}

// Two-product kind, plan_two_product_row: a CTA = one (inv1, inv2) pair x 128 cash levels; cash-independent terms shared
// through shared memory.
int launch_two_product_row(sdpb_handle* h, int t, const double* Vn, double* Vt, int* Qt, long long lo, long long hi) {
    const int Dt = h->pmf_len[t - 1];
    const int segs = (h->dm.nW + 127) / 128;
    const long long pair0 = lo / h->dm.nW, pair1 = (hi - 1) / h->dm.nW;
    const unsigned blocks = (unsigned)((pair1 - pair0 + 1) * segs);
    const size_t smem = (size_t)Dt * sizeof(TwoProductRowTables);
    cudaError_t e = cudaSuccess;
    auto k = t == h->m.T ? bi_two_product_row<true> : bi_two_product_row<false>;
    if (smem > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) k<<<blocks, 128, smem, h->stream>>>(h->dm, t, Dt, h->pmf_off[t - 1], Vn, Vt, Qt, lo, hi, pair0, segs);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return SDPB_ERR_CUDA; }
    return SDPB_OK;
}

size_t staged_smem(int D) { return (size_t)D * 16 + (size_t)8 * D * sizeof(StagedRow); }

// Staged warp-per-state kernel for backorder lead-time models.
template <bool DEDUP>
int launch_staged(sdpb_handle* h, int t, const double* Vn, double* Vt, int* Qt, long long lo, long long hi) {
    const long long n = hi - lo;
    if (n <= 0) return SDPB_OK;
    const int D = h->pmf_len[t - 1];
    const size_t smem = staged_smem(D);
    long long blocks = (n + 7) / 8;
    if (h->dm.lead == 2 && !DEDUP) {  // CTA = 8 consecutive preQ1 of one (x, preQ2): see the kernel
        const long long per_x = (long long)h->dm.nQ * h->dm.nQ;
        const long long rows = (hi - 1) / per_x - lo / per_x + 1;
        blocks = rows * ((h->dm.nQ + 7) / 8) * h->dm.nQ;
    }
    cudaError_t e = cudaSuccess;
    auto k = h->dm.is_min ? bi_backorder_staged<true, DEDUP> : bi_backorder_staged<false, DEDUP>;
    if (smem > 48 * 1024) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) k<<<(unsigned)blocks, 256, smem, h->stream>>>(h->dm, t, D, h->pmf_off[t - 1], Vn, Vt, Qt, lo, hi);
    if (e != cudaSuccess) { h->err = cudaGetErrorString(e); return SDPB_ERR_CUDA; }
    return SDPB_OK;
}

template <int KIND>
void launch_expand(sdpb_handle* h, double* Vt, int* Qt) {
    const long long n = h->hi - h->lo;
    if (n <= 0) return;
    expand_dedup<KIND><<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->dm, h->dHv, h->dHa, Vt, Qt, h->lo, h->hi);
}

template <int KIND, bool SURV>
void launch_reach(sdpb_handle* h, int t) {
    const long long blocks = (h->S + 255) / 256;
    reach_forward<KIND, SURV><<<(unsigned)blocks, 256, 0, h->stream>>>(
        h->dm, t, h->pmf_len[t - 1], h->pmf_off[t - 1], h->dMask[t - 1], t < h->m.T ? h->dMask[t] : nullptr,
        h->dCounters);
}

// Evaluations actually executed for one period in dedup mode (virtual states only).
double count_evals_virtual(const sdpb_handle* h, int t) {
    const sdpb_model& m = h->m;
    const DevModel& d = h->dm;
    const double D = h->pmf_len[t - 1];
    if ((m.flags & SDPB_F_NO_ORDER_LAST) && t == m.T) return (double)h->vS * D;
    if (!(m.flags & SDPB_F_CASH_LIMITED_ACTIONS)) return (double)h->vS * (m.max_order_idx + 1) * D;
    const double v = m.vari_cost_t ? m.vari_cost_t[t - 1] : m.vari_cost;
    const double res = m.reserve_t ? m.reserve_t[t - 1] : 0.0;
    double per_w = 0;
    for (int iw = 0; iw < d.nW; iw++) {
        const double w = cash_of_k(h, d.kmin + iw);
        per_w += (int)std::min((double)m.max_order_idx, std::max(0.0, ((w - res) - m.reserve2) / v)) + 1;
    }
    return per_w * (double)(h->vS / d.nW) * D;
}

// policy table as order quantities (doubles), converted on the device so the host copy is one memcpy
__global__ void policy_to_double(const int* __restrict__ q, double* __restrict__ out, long long n, double step,
                                 int xr, double inv_min, long long stride_x, long long first) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int qi = q[i];
    double v = 0.0;  // bestOrderQty stays 0 when nothing beat the initial value
    if (qi >= 0) v = xr ? (inv_min + (double)((first + i) / stride_x) * step) + (double)qi * step : (double)qi * step;
    out[i] = v;
}

__global__ void gather_vq(const long long* __restrict__ idx, int n, const double* __restrict__ V,
                          const int* __restrict__ Q, double* __restrict__ v, int* __restrict__ q) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { v[i] = V[idx[i]]; q[i] = Q[idx[i]]; }
}

// ---- multi-GPU exchange ----------------------------------------------------------------------------------------
// After the kernels of period t a shard copies the rows of its block that a peer reads into the peer's V_t
// (cudaMemcpyAsync into peer-mapped memory: NVLink), then peer_signal stores the exchange count into the peer's
// flag word; before period t-1 peer_wait spins on this shard's own flag words until every peer it reads from has
// done the same.  Everything is stream-ordered on the device; the host never waits inside a solve.
__global__ void peer_signal(unsigned* const* targets, int n, unsigned epoch) {
    const int i = threadIdx.x;
    if (i >= n) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(targets[i]), "r"(epoch) : "memory");
}

// flags[r] counts the exchanges rank r has completed into this shard.  A peer that never arrives must not hang the
// GPU: after `timeout_ns` the kernel gives up and records which rank was missing in flags[kMaxPeers].
__global__ void peer_wait(unsigned* flags, const int* from, int n, unsigned epoch, unsigned long long timeout_ns) {
    const int i = threadIdx.x;
    if (i >= n) return;
    unsigned* f = flags + from[i];
    unsigned long long t0 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        unsigned v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if ((int)(v - epoch) >= 0) break;
        if (*(volatile unsigned*)(flags + kMaxPeers) != 0) break;  // an earlier wait already failed: do not wait again
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > timeout_ns) { atomicExch(flags + kMaxPeers, 1u + (unsigned)from[i]); break; }
        __nanosleep(256);
    }
}

uint64_t model_hash(const sdpb_handle* h) {  // shards must describe the same model: a cheap fingerprint
    uint64_t x = 1469598103934665603ull;
    auto mix = [&](const void* p, size_t n) {
        const unsigned char* b = (const unsigned char*)p;
        for (size_t i = 0; i < n; i++) { x ^= b[i]; x *= 1099511628211ull; }
    };
    const sdpb_model& m = h->m;
    mix(&m.cost_kind, sizeof(int32_t) * 7);
    mix(&m.gamma, sizeof(double));
    mix(&m.inv_min, sizeof(double) * 5);
    mix(&m.fixed_cost, sizeof(double) * 14);
    mix(h->pmf_len.data(), h->pmf_len.size() * sizeof(int));
    mix(h->pmf_d.data(), h->pmf_d.size() * sizeof(double));
    mix(h->pmf_p.data(), h->pmf_p.size() * sizeof(double));
    return x;
}

int solve_period(sdpb_handle* h, int t);

// One period of a sharded solve: kernels, then (t > 1) the pushes and the flag.  `wait_now`: also enqueue the wait for
// the peers' rows (a group driven by one host thread enqueues every shard's pushes first, then every shard's wait).
int enqueue_period_exchange_wait(sdpb_handle* h) {
    PeerLink& P = h->peer;
    if (P.by_events) {
        for (int r : P.recv_from) CU(cudaStreamWaitEvent(h->stream, P.peer_handles[r]->peer.ev_pushed, 0));
        return SDPB_OK;
    }
    if (!P.recv_from.empty()) {
        peer_wait<<<1, kMaxPeers, 0, h->stream>>>(reinterpret_cast<unsigned*>(h->slab), P.d_from, (int)P.recv_from.size(),
                                                  P.epoch, 20ull * 1000000000ull);
        CU(cudaGetLastError());
    }
    return SDPB_OK;
}

int enqueue_period_sharded(sdpb_handle* h, int t, bool wait_now) {
    PeerLink& P = h->peer;
    const bool prof = !h->prof_ev.empty();
    cudaEvent_t* ev = prof ? h->prof_ev.data() + 4 * (size_t)(t - 1) : nullptr;
    if (prof) CU(cudaEventRecord(ev[0], h->stream));
    h->push_fused = false;
    int rc = solve_period(h, t);
    if (rc != SDPB_OK) return rc;
    if (prof) CU(cudaEventRecord(ev[1], h->stream));
    if (t > 1) {  // V_1 is read by nobody
        P.epoch++;
        if (!h->push_fused) for (const PeerSend& sd : P.sends) {
            const PeerInfo& pi = P.info[sd.rank];
            char* dst = P.mapped[sd.rank] + pi.v_off0 + (size_t)(t - 1) * pi.v_stride + (size_t)(sd.a - pi.vlo) * sizeof(double);
            CU(cudaMemcpyAsync(dst, h->dV[t - 1] + sd.a, (size_t)(sd.b - sd.a) * sizeof(double), cudaMemcpyDefault, h->stream));
        }
        if (P.by_events) {
            CU(cudaEventRecord(P.ev_pushed, h->stream));
        } else if (!P.sends.empty()) {
            peer_signal<<<1, kMaxPeers, 0, h->stream>>>(P.d_targets, (int)P.sends.size(), P.epoch);
            CU(cudaGetLastError());
        }
        if (prof) CU(cudaEventRecord(ev[2], h->stream));
        if (wait_now) {
            rc = enqueue_period_exchange_wait(h);
            if (rc != SDPB_OK) return rc;
            if (prof) CU(cudaEventRecord(ev[3], h->stream));
        }
    } else if (prof) {
        CU(cudaEventRecord(ev[2], h->stream));
        CU(cudaEventRecord(ev[3], h->stream));
    }
    return SDPB_OK;
}

// After the stream has drained: did a wait give up?  Fill the per-period profile.
int finish_sharded(sdpb_handle* h) {
    unsigned errw = 0;
    if (!h->peer.by_events) CU(cudaMemcpy(&errw, h->slab + kMaxPeers * sizeof(unsigned), sizeof errw, cudaMemcpyDeviceToHost));
    if (errw) {
        h->err = "shard " + std::to_string(errw - 1) + " did not deliver its rows of V_t within 20 s";
        return SDPB_ERR_PEER;
    }
    if (!h->prof_ev.empty()) {
        h->prof_ms.assign(3 * (size_t)h->m.T, 0.0);
        double ex = 0;
        for (int t = 1; t <= h->m.T; t++) {
            cudaEvent_t* ev = h->prof_ev.data() + 4 * (size_t)(t - 1);
            for (int k = 0; k < 3; k++) {
                float ms = 0;
                if (cudaEventElapsedTime(&ms, ev[k], ev[k + 1]) != cudaSuccess) { cudaGetLastError(); ms = 0; }
                h->prof_ms[3 * (size_t)(t - 1) + k] = ms;
                if (k > 0) ex += ms;
            }
        }
        h->stats.exchange_ms = ex;
    }
    return SDPB_OK;
}

// Scratch for action slices: a (value, action) entry per slice and state (a smaller earlier one stays in dev_allocs).
int grow_slice_scratch(sdpb_handle* h, size_t need, double*& v, int*& a, size_t& cap) {
    if (need <= cap) return SDPB_OK;
    void* p = nullptr;
    CU(dev_alloc(h, &p, need * sizeof(double)));
    v = (double*)p;
    CU(dev_alloc(h, &p, need * sizeof(int)));
    a = (int*)p;
    cap = need;
    return SDPB_OK;
}

// Runs the kernel family choose_period_kernel picked for period t, and counts it in h->stats.
int solve_period(sdpb_handle* h, int t) {
    const sdpb_model& m = h->m;
    if (t < 1 || t > m.T) { h->err = "period out of range"; return SDPB_ERR_ARG; }
    if (t < m.T && !h->solved[t]) { h->err = "period t+1 not solved yet"; return SDPB_ERR_STATE; }
    // V_{t+1}: the next period's table, or in period T the boundary table when the model has one
    // (CashRecursionV.java:125-128), else nothing (Recursion.java:140)
    const double* Vn = t < m.T ? h->dV[t] : h->dTerm;
    const bool last = Vn == nullptr;
    const int D = h->pmf_len[t - 1], off = h->pmf_off[t - 1];
    const bool plain = (m.flags & SDPB_F_NO_ORDER_LAST) && t == m.T;  // A(s) = {0}: see choose_period_kernel
    const bool surv = m.recursion == SDPB_REC_SURVIVAL;
    // dedup (lead-time models): solve each distinct (x + preQ, ...) of the virtual grid once, then broadcast (exact)
    double* Vt = h->dedup ? h->dHv : h->dV[t - 1];
    int* Qt = h->dedup ? h->dHa : h->dQ[t - 1];
    const long long lo = h->dedup ? 0 : h->lo, hi = h->dedup ? h->vS : h->hi;
    const double ev_range = (double)(hi - lo) * (m.max_order_idx + 1) * D;  // every action of every state of [lo, hi)
    double executed = h->dedup ? count_evals_virtual(h, t) : count_evals_period(h, t);
    const bool push = h->peer.attached && t > 1 && !h->peer.sends.empty();  // a peer reads rows of this period
    const sdpb_kernel_choice kind = h->period_kernel[t - 1];
    sdpb_kernel_choice used = kind;
    int rc = SDPB_OK;
    switch (kind) {
    case SDPB_KERNEL_COLLAPSED: {  // opt-in, not bit-identical (kernel_collapsed.cuh)
        rc = launch_collapsed(h->dm, t, D, off, Vn, h->dLc, h->lc_il0, h->dG, Vt, Qt, h->stream);
        if (rc != SDPB_OK) { h->err = "collapsed kernel launch failed"; return rc; }
        const double nY = (double)h->dm.nI + m.max_order_idx, nA = m.max_order_idx + 1.0;
        h->stats.launches++;                     // (two kernels)
        executed = nY * D + (double)h->S * nA;   // level-demand pairs + state-action pairs
        h->stats.fp64_ops += nY * D * (Vn ? 7.0 : 5.0) + (double)h->S * nA * 3.0;
        break;
    }
    case SDPB_KERNEL_TILED: {
        int variant = 1;
        rc = launch_tiled(h->tiled, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream, &variant);
        if (rc != SDPB_OK) { h->err = "tiled kernel launch failed"; return rc; }
        if (variant == 2) {
            used = SDPB_KERNEL_TILED2;
            // per 16 evaluations: 4 new costs + 4 products + 16 * (mul, add, add); last period: 4 + 16 * 2
            h->stats.fp64_ops += last ? ev_range * 2.25 : ev_range * 3.5;
        } else {
            // per evaluation add+mul+add(+add), plus one mul per R evaluations
            h->stats.fp64_ops += last ? ev_range * 3.0 : ev_range * 4.0 + ev_range / kTiledR;
        }
        break;
    }
    case SDPB_KERNEL_CASH_DIAG:
    case SDPB_KERNEL_CASH_INT: {
        const bool diag = kind == SDPB_KERNEL_CASH_DIAG;
        const CashIntShape sh = cash_int_shape(m, h->dm, t, lo, hi, h->sm_count);
        const int parts = diag ? cash_diag_parts(m, h->dm, h->cash.period[t - 1], lo, hi, h->sm_count) : sh.parts;
        if (int e = grow_slice_scratch(h, parts > 1 ? (size_t)parts * (size_t)(hi - lo) : 0, h->cash.slice_v,
                                       h->cash.slice_a, h->cash.slice_cap))
            return e;
        // a sliced launch: merge_action_slices also stores the rows the peers read
        const DevPeer* d_peers = push ? (const DevPeer*)h->peer.d_peers : nullptr;
        const int n_peers = push ? (int)h->peer.sends.size() : 0;
        rc = diag ? launch_cash_diag(h->cash, parts, m, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream, d_peers, n_peers)
                  : launch_cash(h->cash, sh, m, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream, d_peers, n_peers);
        if (rc != SDPB_OK) { h->err = "cash kernel launch failed"; return rc; }
        if (parts > 1) {
            h->stats.launches++;  // merge_action_slices
            if (push) h->push_fused = true;
        }
        if (diag) h->stats.fp64_ops += executed * (surv ? 2.0 : 3.0 + 2.0 / kDiagYT);
        else if (t == m.T) h->stats.fp64_ops += executed * (surv ? 2.0 + 3.0 / kCashR : 1.0 + 4.0 / (sh.wide ? kCashRLast : kCashR));
        else h->stats.fp64_ops += executed * (surv ? 2.0 : 3.0 + 2.0 / kCashR);
        break;
    }
    case SDPB_KERNEL_LEAD_Q2: {
        const Q2Plan qp = plan_q2(m, h->dm, D, h->pmf_di.data() + off);
        const Q2Shape shape = q2_shape(qp, h->dm, D, lo, hi, h->sm_count);
        int64_t rlo = 0, rhi = h->S;
        sdpb_shard_reads(h, &rlo, &rhi);
        const long long per_x = (long long)h->dm.nQ * h->dm.nQ;
        // multi-GPU: the kernel's epilogue stores the rows its (at most two) neighbours read straight into their
        // tables, or, when the action range is cut over separate CTAs, merge_action_slices does; enqueue_period_sharded
        // then skips the copies
        PeerStore ps[kQ2MaxPeers];
        int nps = 0;
        if (shape.slices > 1) {
            if (int e = grow_slice_scratch(h, (size_t)shape.slices * (size_t)(hi - lo), h->q2_slice_v, h->q2_slice_a,
                                           h->q2_slice_cap))
                return e;
            if (push) h->push_fused = true;
        } else if (push && h->peer.sends.size() <= (size_t)kQ2MaxPeers) {
            for (const PeerSend& sd : h->peer.sends) {
                const PeerInfo& pi = h->peer.info[sd.rank];
                char* base = h->peer.mapped[sd.rank] + pi.v_off0 + (size_t)(t - 1) * pi.v_stride;
                ps[nps++] = PeerStore{reinterpret_cast<double*>(base) - pi.vlo, sd.a, sd.b};
            }
            h->push_fused = true;
        }
        const bool merge_pushes = push && shape.slices > 1;
        rc = launch_q2(qp, shape, h->dm, t, D, off, Vn, h->dVT, Vt, Qt, lo, hi, (int)(rlo / per_x), (int)(rhi / per_x),
                       h->stream, ps, nps, h->q2_slice_v, h->q2_slice_a, h->q2_slice_cap,
                       merge_pushes ? (const DevPeer*)h->peer.d_peers : nullptr, merge_pushes ? (int)h->peer.sends.size() : 0);
        if (rc != SDPB_OK) return rc;
        const bool ran = hi > lo;  // (an empty shard launches nothing and reports bi_lead_q2)
        if (!last) h->stats.launches++;                      // the transposition pass
        if (ran && shape.slices > 1) h->stats.launches++;    // merge_action_slices
        // per evaluation: (mul, add, mul, add) + one cost per 8 -- or, with the products p*(fv + L) shared by the CTA
        // (bi_lead_q2m), (add, mul, add); the last period has no continuation term
        if (ran && shape.shared) { used = SDPB_KERNEL_LEAD_Q2M; h->stats.fp64_ops += ev_range * (last ? 1.0 : 3.0); }
        else h->stats.fp64_ops += ev_range * (last ? (1.0 + 2.0 * kQ2YT) / kQ2YT : (1.0 + 4.0 * kQ2YT) / kQ2YT);
        break;
    }
    case SDPB_KERNEL_LEAD_COL: {
        const ColPlan cp = plan_col(m, h->dm, D, h->pmf_di.data() + off, h->dedup);
        rc = h->dedup ? launch_col<true>(cp, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream)
                      : launch_col<false>(cp, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream);
        // per YT evaluations: 1 new cost + YT (p*c) + YT adds (+ YT (p*gamma*V) + YT adds)
        h->stats.fp64_ops += ev_range * (last ? (1.0 + 2.0 * kColYT) / kColYT : (1.0 + 4.0 * kColYT) / kColYT);
        break;
    }
    case SDPB_KERNEL_LEAD_SLAB: {
        const LeadPlan lp = plan_lead(m, h->dm, D, h->pmf_di.data() + off);
        rc = h->dedup ? launch_lead<true>(lp, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream)
                      : launch_lead<false>(lp, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream);
        const double q = 4.0 * lp.RQ;  // evaluations per thread per demand point
        h->stats.fp64_ops += ev_range * (last ? (5.0 + q) / q : (5.0 + 3.0 * q) / q);
        break;
    }
    case SDPB_KERNEL_STAGED:
        rc = h->dedup ? launch_staged<true>(h, t, Vn, Vt, Qt, lo, hi) : launch_staged<false>(h, t, Vn, Vt, Qt, lo, hi);
        // per evaluation: add, mul, add (+ mul, add when a continuation exists)
        h->stats.fp64_ops += (double)(hi - lo) * (plain ? 1 : m.max_order_idx + 1) * D * (last ? 3.0 : 5.0);
        break;
    case SDPB_KERNEL_CASH_TAIL: {
        const CashTailPlan tp = plan_cash_tail(m, h->dm, D, h->pmf_d.data(), (int)h->pmf_d.size());
        rc = launch_cash_tail(tp, m, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream);
        // DADD + DMUL per evaluation as counted by ncu (profiles/r02_fp64_audit.md)
        const int kd = m.cost_kind;  // (overdraft-limit / -testing: a few more for the two interest products)
        const double body = kd == SDPB_COST_CASH_DEPOSIT ? 4.0 : kd == SDPB_COST_CASH_OVERDRAFT ? 2.0 : kd == SDPB_COST_CASH_OD_LIMIT ? 9.0 : 7.0;
        h->stats.fp64_ops += executed * (last ? body + 3.0 : body + 8.0);
        break;
    }
    case SDPB_KERNEL_CASH_ROW:
        rc = launch_cash_row(m, h->dm, t, D, off, Vn, Vt, Qt, lo, hi, h->stream);
        // cash-dependent tail per evaluation: deposit chain 4, salvage 1, end cash 1, p*c 2 (+ clamp / quantiser /
        // continuation 5 when a successor exists); compares and selects not counted
        h->stats.fp64_ops += executed * (last ? 8.0 : 13.0);
        break;
    case SDPB_KERNEL_TWO_PRODUCT_ROW:
        rc = launch_two_product_row(h, t, Vn, Vt, Qt, lo, hi);
        h->stats.fp64_ops += executed * (t == m.T ? 1.0 : 3.0);
        break;
    default: {  // SDPB_KERNEL_GENERIC
        rc = h->dedup ? dispatch_generic_d<true>(h, t, Vn, Vt, Qt, lo, hi) : dispatch_generic_d<false>(h, t, Vn, Vt, Qt, lo, hi);
        // bi_generic evaluates the lambdas as written: its fp64 count per evaluation is MEASURED (ncu DADD + DMUL thread
        // instructions, profiles/r02_fp64_audit.md), not derived; kinds that were not measured report nothing
        double per_eval = 0.0;
        switch (m.cost_kind) {
        case SDPB_COST_BACKORDER: per_eval = 8.4; break;
        case SDPB_COST_CASH_DEPOSIT: per_eval = 18.4; break;
        case SDPB_COST_CASH_OVERDRAFT: per_eval = 11.5; break;
        case SDPB_COST_STAFF: per_eval = 7.4; break;
        default: break;
        }
        h->stats.fp64_ops += per_eval * executed;
        break;
    }
    }
    if (rc != SDPB_OK) return rc;
    if (h->dedup) {
        switch (m.cost_kind) {
        case SDPB_COST_BACKORDER: launch_expand<SDPB_COST_BACKORDER>(h, h->dV[t - 1], h->dQ[t - 1]); break;
        case SDPB_COST_CASH_DEPOSIT: launch_expand<SDPB_COST_CASH_DEPOSIT>(h, h->dV[t - 1], h->dQ[t - 1]); break;
        default: launch_expand<SDPB_COST_CASH_OVERDRAFT>(h, h->dV[t - 1], h->dQ[t - 1]); break;
        }
        h->stats.launches++;
    }
    CU(cudaGetLastError());
    h->solved[t - 1] = 1;
    h->stats.launches++;
    h->stats.evals += count_evals_period(h, t);  // what the reference evaluates
    h->stats.evals_executed += executed;
    // The kernel a solve reports: the last one that ran, except that GENERIC does not replace a specialised kernel of
    // an earlier period, and CASH_INT (period T) does not replace CASH_DIAG.
    const int prev = h->stats.kernel_used;
    if (!(used == SDPB_KERNEL_GENERIC && prev != 0) && !(used == SDPB_KERNEL_CASH_INT && prev == SDPB_KERNEL_CASH_DIAG))
        h->stats.kernel_used = used;
    return SDPB_OK;
}

// The kernel family that solves period t, fixed by sdpb_create from the model, the request (opt.kernel), dedup, the
// per-period plans, the shard's range and whether dVT exists.  "plain": period T of an SDPB_F_NO_ORDER_LAST model (A(s)
// = {0}, SingleProductLeadtime.java:74-75, a rule only decode_state() knows); "term_T": period T with a boundary table
// (the integer cash kernels fold "last period" and "no continuation" into one flag).  The first rule that applies wins:
//   request COLLAPSED or GENERIC: that kernel
//   backorder, lead 0, clamp: TILED (tiled / tiled2 at launch) if the period has a plan and is not plain
//   integer-exact deposit models, any request, periods with a plan, not plain or term_T, a non-empty shard:
//     CASH_DIAG if t < T, the request is not CASH_INT and cash_diag_ok;  CASH_INT if its tables fit
//   backorder, lead >= 1, not plain: LEAD_Q2 (q2 / q2m at launch) if dVT exists (lead 2, unfolded, request AUTO or
//     LEAD_Q2) and plan_q2 holds;  LEAD_COL if the request is neither STAGED nor LEAD_SLAB and plan_col holds;
//     LEAD_SLAB if the request is not STAGED and plan_lead holds
//   backorder, lead >= 1: STAGED if its tables fit
//   cash kinds with row-shared kernels, lead 0: CASH_TAIL if the request is not CASH_ROW and plan_cash_tail holds;
//     CASH_ROW if cash_row_ok
//   two-product: TWO_PRODUCT_ROW in a non-empty shard, not term_T, if plan_two_product_row holds
//   otherwise GENERIC
// So a CASH_ROW request on an integer-exact deposit model runs the integer cash kernels, and a TILED request on a
// backorder lead-time model runs LEAD_COL.
sdpb_kernel_choice choose_period_kernel(const sdpb_handle* h, int t) {
    const sdpb_model& m = h->m;
    const int K = h->opt.kernel;
    if (K == SDPB_KERNEL_COLLAPSED || K == SDPB_KERNEL_GENERIC) return (sdpb_kernel_choice)K;
    const int D = h->pmf_len[t - 1];
    const int* di = h->pmf_di.data() + h->pmf_off[t - 1];
    const bool plain = (m.flags & SDPB_F_NO_ORDER_LAST) && t == m.T;
    const bool term_T = t == m.T && h->dTerm != nullptr;
    const bool backorder_lead = m.cost_kind == SDPB_COST_BACKORDER && m.lead_time >= 1;
    if (h->tiled.available && !plain && (h->tiled.period[t - 1].ok || h->tiled.period[t - 1].ok2))
        return SDPB_KERNEL_TILED;
    if (h->cash.available && h->cash.period[t - 1].ok && !plain && !term_T && h->hi > h->lo) {
        if (K != SDPB_KERNEL_CASH_INT && t < m.T && cash_diag_ok(h->cash.period[t - 1], m, h->dm, D))
            return SDPB_KERNEL_CASH_DIAG;
        if (cash_int_smem(D) <= 200 * 1024) return SDPB_KERNEL_CASH_INT;
    }
    if (backorder_lead && !plain) {
        if (h->dVT && plan_q2(m, h->dm, D, di).ok) return SDPB_KERNEL_LEAD_Q2;
        if (K != SDPB_KERNEL_STAGED && K != SDPB_KERNEL_LEAD_SLAB && plan_col(m, h->dm, D, di, h->dedup).ok)
            return SDPB_KERNEL_LEAD_COL;
        if (K != SDPB_KERNEL_STAGED && plan_lead(m, h->dm, D, di).ok) return SDPB_KERNEL_LEAD_SLAB;
    }
    if (backorder_lead && staged_smem(D) <= 200 * 1024) return SDPB_KERNEL_STAGED;
    if (K != SDPB_KERNEL_CASH_ROW && plan_cash_tail(m, h->dm, D, h->pmf_d.data(), (int)h->pmf_d.size()).ok)
        return SDPB_KERNEL_CASH_TAIL;
    if (cash_row_ok(m, h->dm, D)) return SDPB_KERNEL_CASH_ROW;
    if (two_product(m) && h->hi > h->lo && !term_T && plan_two_product_row(m, h->dm, t, D))
        return SDPB_KERNEL_TWO_PRODUCT_ROW;
    return SDPB_KERNEL_GENERIC;
}

}  // namespace

extern "C" {

int sdpb_abi_version(void) { return SDPB_ABI_VERSION; }
size_t sdpb_sizeof_model(void) { return sizeof(sdpb_model); }
size_t sdpb_sizeof_options(void) { return sizeof(sdpb_options); }
size_t sdpb_sizeof_grid(void) { return sizeof(sdpb_grid); }
size_t sdpb_sizeof_stats(void) { return sizeof(sdpb_stats); }

const char* sdpb_last_error(const sdpb_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

static void forget_batches_of(sdpb_handle* h);

void sdpb_destroy(sdpb_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    forget_batches_of(h);  // a captured batch graph must not outlive one of its handles
    if (h->stream) cudaStreamSynchronize(h->stream);  // (peers may still be reading flags this stream raises)
    if (h->stream) for (void* p : h->dev_allocs) cudaFreeAsync(p, h->stream);
    free_tiled(h->tiled);
    // (peers' slabs mapped through CUDA IPC stay mapped: ipc_map caches them for the next handle)
    if (h->slab) slab_release(h->device, h->slab, h->slab_bytes);
    if (h->peer.ev_pushed) cudaEventDestroy(h->peer.ev_pushed);
    for (cudaEvent_t e : h->prof_ev) if (e) cudaEventDestroy(e);
    if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->own_stream && h->stream) { cudaStreamSynchronize(h->stream); cudaStreamDestroy(h->stream); }
    cudaGetLastError();
    delete h;
}

int sdpb_create(const sdpb_model* m, const sdpb_options* opt, sdpb_handle** out) {
    g_create_error.clear();
    // SDPB_TRACE=1: wall-clock checkpoints of this call on stderr
    static const bool trace = std::getenv("SDPB_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto mark = [&](const char* what) {
        if (trace)
            std::fprintf(stderr, "[sdpb_create] %-18s %8.3f ms\n", what,
                         std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count());
    };
    if (!m || !out) return fail_create(nullptr, SDPB_ERR_ARG, "null argument");
    *out = nullptr;
    if (m->struct_size != sizeof(sdpb_model))
        return fail_create(nullptr, SDPB_ERR_ARG, "sdpb_model.struct_size does not match this library");
    if (opt && opt->struct_size != sizeof(sdpb_options))
        return fail_create(nullptr, SDPB_ERR_ARG, "sdpb_options.struct_size does not match this library");
    if (m->T < 1 || !m->pmf_len || !m->pmf_d || !m->pmf_p)
        return fail_create(nullptr, SDPB_ERR_ARG, "T < 1 or null pmf");
    if (m->cost_kind < 0 || m->cost_kind > SDPB_COST_STAFF) return fail_create(nullptr, SDPB_ERR_ARG, "bad cost_kind");
    if (m->cost_kind == SDPB_COST_STAFF &&
        (!m->apmf_len || !m->apmf_p || !m->min_level_t || m->step != 1.0 || m->lead_time != 0 ||
         m->recursion != SDPB_REC_EXPECT))
        return fail_create(nullptr, SDPB_ERR_ARG, "staff kind needs apmf_len, apmf_p, min_level_t and a unit step");
    if (m->cost_kind == SDPB_COST_CASH_TWO_PRODUCT &&
        (!m->pmf_d2 || m->quantiser != SDPB_Q_TRUNC || m->recursion != SDPB_REC_EXPECT || m->step != 1.0))
        return fail_create(nullptr, SDPB_ERR_ARG, "two-product kind needs pmf_d2, the (int) cash quantiser, unit step");
    if (m->cost_kind >= SDPB_COST_CASH_OD_LIMIT && m->lead_time != 0)
        return fail_create(nullptr, SDPB_ERR_ARG, "this cost kind has no lead-time variant in the reference");
    if (m->lead_time < 0 || m->lead_time > 2) return fail_create(nullptr, SDPB_ERR_ARG, "lead_time must be 0, 1 or 2");
    if (m->cost_kind == SDPB_COST_CASH_XR && m->lead_time != 0)
        return fail_create(nullptr, SDPB_ERR_ARG, "XR kind has no lead time");
    if (m->recursion == SDPB_REC_SURVIVAL &&
        !(m->cost_kind == SDPB_COST_CASH_DEPOSIT || m->cost_kind == SDPB_COST_CASH_OVERDRAFT))
        return fail_create(nullptr, SDPB_ERR_ARG, "survival recursion needs a cash kind");
    if (m->max_order_idx < 0) return fail_create(nullptr, SDPB_ERR_ARG, "max_order_idx < 0");
    if (m->terminal_value && m->recursion == SDPB_REC_SURVIVAL)
        return fail_create(nullptr, SDPB_ERR_ARG, "the survival recursion has its own terminal rule (RiskRecursion.java:80-84)");
    if (m->terminal_value && opt && opt->dedup)
        return fail_create(nullptr, SDPB_ERR_ARG, "a terminal value table need not depend on x + preQ only: dedup is off limits");

    // ---- exact-grid validation: every x, a, d is an integer multiple of a power-of-two step ----
    int ex;
    if (!(m->step > 0) || std::frexp(m->step, &ex) != 0.5)
        return fail_create(nullptr, SDPB_ERR_OFFGRID, "step must be a positive power of two");
    if (!is_int(m->inv_min / m->step) || !is_int(m->inv_max / m->step) || m->inv_max < m->inv_min)
        return fail_create(nullptr, SDPB_ERR_OFFGRID, "inventory bounds are not multiples of step");

    sdpb_handle* h = new (std::nothrow) sdpb_handle();
    if (!h) return fail_create(nullptr, SDPB_ERR_NOMEM, "out of host memory");
    h->m = *m;
    if (opt) h->opt = *opt;
    else { h->opt.struct_size = sizeof(sdpb_options); h->opt.device = -1; h->opt.shard_count = 1; }
    if (h->opt.shard_count < 1) h->opt.shard_count = 1;
    if (h->opt.kernel == SDPB_KERNEL_LEAD_Q2M) h->opt.kernel = SDPB_KERNEL_LEAD_Q2;  // a reported-only name: the library chooses between the two
    if (h->opt.shard_rank < 0 || h->opt.shard_rank >= h->opt.shard_count)
        return fail_create(h, SDPB_ERR_ARG, "shard_rank out of range");

    const int T = m->T;
    h->pmf_len.assign(m->pmf_len, m->pmf_len + T);
    h->pmf_off.assign(T + 1, 0);
    for (int t = 0; t < T; t++) {
        if (h->pmf_len[t] < 1) return fail_create(h, SDPB_ERR_ARG, "empty pmf row");
        h->pmf_off[t + 1] = h->pmf_off[t] + h->pmf_len[t];
    }
    const int NP = h->pmf_off[T];
    h->pmf_d.assign(m->pmf_d, m->pmf_d + NP);
    h->pmf_p.assign(m->pmf_p, m->pmf_p + NP);
    h->m.pmf_len = h->pmf_len.data();
    h->m.pmf_d = h->pmf_d.data();
    h->m.pmf_p = h->pmf_p.data();
    std::vector<double> pg(NP), pd2;
    std::vector<int> pdi(NP), pdi2;
    if (m->cost_kind == SDPB_COST_CASH_TWO_PRODUCT) {
        pd2.assign(m->pmf_d2, m->pmf_d2 + NP);
        pdi2.resize(NP);
        for (int j = 0; j < NP; j++) pdi2[j] = (int)pd2[j];  // new Demands((int) d1, (int) d2)
        h->pmf_d2 = pd2;
        h->m.pmf_d2 = h->pmf_d2.data();
    }
    for (int j = 0; j < NP; j++) {
        double f = h->pmf_d[j] / m->step;
        if (m->cost_kind == SDPB_COST_CASH_TWO_PRODUCT) f = (double)(int)h->pmf_d[j];  // (int) cast in the reference
        if (!is_int(f) || std::fabs(f) > 1e9)
            return fail_create(h, SDPB_ERR_OFFGRID, "a demand value is not a multiple of step");
        pdi[j] = (int)f;
        pg[j] = h->pmf_p[j] * m->gamma;  // first product of `p * gamma * V` (CashRecursion.java:120)
    }
    h->pmf_di = pdi;
    // per-period parameter tables; deep copies so the caller's arrays may go away
    std::vector<double> price_t(T), v_t(T), ovh_t(T), res_t(T);
    for (int t = 0; t < T; t++) {
        price_t[t] = m->price_t ? m->price_t[t] : m->price;
        v_t[t] = m->vari_cost_t ? m->vari_cost_t[t] : m->vari_cost;
        ovh_t[t] = m->overhead_t ? m->overhead_t[t] : m->overhead;
        res_t[t] = m->reserve_t ? m->reserve_t[t] : 0.0;
    }

    mark("validated");
    DevModel& d = h->dm;
    d.cost_kind = m->cost_kind;
    d.recursion = m->recursion;
    d.is_min = (m->recursion == SDPB_REC_SURVIVAL) ? 0 : (m->direction == SDPB_MIN);
    d.T = T;
    d.lead = m->lead_time;
    d.max_order_idx = m->max_order_idx;
    d.flags = m->flags;
    d.quantiser = m->quantiser;
    d.nI = (int)h_jround((m->inv_max - m->inv_min) / m->step) + 1;
    d.nQ = m->lead_time > 0 ? m->max_order_idx + 1 : 1;
    d.i_zero = (int)h_jround((0.0 - m->inv_min) / m->step);
    d.inv_min = m->inv_min;
    d.step = m->step;
    d.nW = 1;
    d.kmin = 0;
    d.q_mul = d.q_div = 1.0;
    d.q_idiv = 1;
    d.q_magic = 0;
    if (has_cash(*m)) {
        if (!(m->q_mul > 0) || !(m->q_div > 0) || m->cash_max < m->cash_min)
            return fail_create(h, SDPB_ERR_ARG, "bad cash axis (q_mul, q_div > 0; cash_max >= cash_min)");
        if (m->quantiser == SDPB_Q_LONGDIV && (!is_int(m->q_div) || m->q_div < 1))
            return fail_create(h, SDPB_ERR_ARG, "SDPB_Q_LONGDIV needs an integer q_div >= 1");
        if (m->quantiser != SDPB_Q_DIV && m->quantiser != SDPB_Q_LONGDIV && m->quantiser != SDPB_Q_TRUNC)
            return fail_create(h, SDPB_ERR_ARG, "bad quantiser");
        long long kmin, kmax;
        if (m->cost_kind == SDPB_COST_CASH_XR) {
            if (m->vari_cost_t) return fail_create(h, SDPB_ERR_ARG, "XR kind takes a constant vari_cost");
            if (!is_int(m->vari_cost * m->step) || m->quantiser != SDPB_Q_LONGDIV || m->q_div != 1.0)
                return fail_create(h, SDPB_ERR_OFFGRID, "XR kind needs integer v*step and the round(w*1)/1 quantiser");
            kmin = h_jround(quantise(*m, m->cash_min) + m->vari_cost * m->inv_min);
            kmax = h_jround(quantise(*m, m->cash_max) + m->vari_cost * m->inv_max);
        } else {
            kmin = cash_k_of(*m, quantise(*m, m->cash_min));
            kmax = cash_k_of(*m, quantise(*m, m->cash_max));
        }
        if (kmax < kmin || kmax - kmin > 100000000ll) return fail_create(h, SDPB_ERR_ARG, "cash axis too large");
        d.kmin = kmin;
        d.nW = (int)(kmax - kmin + 1);
        d.q_mul = m->q_mul;
        d.q_div = m->q_div;
        d.q_idiv = (long long)m->q_div;
        d.q_magic = (d.q_idiv >= 2 && d.q_idiv < 32768) ? ((1ull << 47) + (unsigned long long)d.q_idiv - 1) / (unsigned long long)d.q_idiv : 0;
    }
    d.cash_min = m->cash_min;
    d.cash_max = m->cash_max;
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
    d.price2 = m->price2; d.v2 = m->vari_cost2; d.salvage2 = m->salvage2; d.tie_tol = m->tie_tolerance;
    d.pmf_d2 = nullptr; d.pmf_di2 = nullptr;
    d.apmf_len = nullptr; d.apmf_off = nullptr; d.apmf_p = nullptr; d.min_level_t = nullptr;
    long long S = d.nI;
    if (two_product(*m)) S *= d.nI;
    for (int l = 0; l < m->lead_time; l++) S *= d.nQ;
    S *= d.nW;
    d.S = S;
    h->S = S;
    {   // 32-bit successor arithmetic (successor32): every index and quantised cash value below 2^30
        const double cmax = std::max(std::fabs(m->cash_min), std::fabs(m->cash_max));
        const double qm = std::max(1.0, std::fabs(m->q_mul));
        double vmax = std::fabs(m->vari_cost);
        for (double v : v_t) vmax = std::max(vmax, std::fabs(v));
        const double xr = m->cost_kind == SDPB_COST_CASH_XR
                              ? vmax * std::max(std::fabs(m->inv_min), std::fabs(m->inv_max)) : 0.0;
        d.small = (S < (1ll << 30) && (cmax + xr + 1.0) * qm < 1073741824.0 &&
                   std::llabs(d.kmin) < (1ll << 30) && d.q_idiv < (1ll << 30)) ? 1 : 0;
    }
    h->ndim = 1 + (two_product(*m) ? 1 : 0) + (has_cash(*m) ? 1 : 0) + m->lead_time;
    const long long chunk = (S + h->opt.shard_count - 1) / h->opt.shard_count;
    h->Spad = chunk * h->opt.shard_count;
    h->lo = std::min(S, chunk * h->opt.shard_rank);
    h->hi = std::min(S, h->lo + chunk);

    // ---- device ----
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail_create(h, SDPB_ERR_NO_DEVICE, "no CUDA device (libsdpb200 has no CPU path)");
    int dev = h->opt.device;
    if (dev < 0) cudaGetDevice(&dev);
    if (dev >= ndev) return fail_create(h, SDPB_ERR_NO_DEVICE, "device ordinal out of range");
    h->device = dev;
    // two attribute queries instead of cudaGetDeviceProperties, which costs 3-30 ms per call
    int cc_major = 0, sm_count = 0;
    if (cudaSetDevice(dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return fail_create(h, SDPB_ERR_NO_DEVICE, "cannot select CUDA device");
    if (cc_major != 10)
        return fail_create(h, SDPB_ERR_NO_DEVICE, "libsdpb200 is built for sm_100a (B200) only");
    mark("device selected");
    if (h->opt.stream) { h->stream = (cudaStream_t)h->opt.stream; }
    else {
        if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess)
            return fail_create(h, SDPB_ERR_CUDA, "cudaStreamCreate failed");
        h->own_stream = true;
    }
    cudaEventCreate(&h->ev0);
    cudaEventCreate(&h->ev1);
    mark("stream, events");

    double *dp = nullptr;
    int* di = nullptr;
    int rc;
#define UP(vec, field, tmp) \
    if ((rc = upload(h, vec, &tmp)) != SDPB_OK) return fail_create(h, rc, h->err); \
    d.field = tmp;
    UP(price_t, price_t, dp) UP(v_t, v_t, dp) UP(ovh_t, ovh_t, dp) UP(res_t, reserve_t, dp)
    UP(h->pmf_d, pmf_d, dp) UP(h->pmf_p, pmf_p, dp) UP(pg, pmf_pg, dp) UP(pdi, pmf_di, di)
    {
        std::vector<double> rec((size_t)4 * NP);
        for (int j = 0; j < NP; j++) {
            rec[4 * (size_t)j] = h->pmf_d[j];
            rec[4 * (size_t)j + 1] = h->pmf_p[j];
            rec[4 * (size_t)j + 2] = pg[j];
            const long long bits = (long long)(unsigned)pdi[j];  // read back with __double2loint
            std::memcpy(&rec[4 * (size_t)j + 3], &bits, sizeof bits);
        }
        if ((rc = upload(h, rec, &dp)) != SDPB_OK) return fail_create(h, rc, h->err);
        d.pmf_rec = reinterpret_cast<const double2*>(dp);
    }
    if (two_product(*m)) { UP(pd2, pmf_d2, dp) UP(pdi2, pmf_di2, di) }
    if (staff_kind(*m)) {
        const size_t rows = (size_t)T * d.nI;
        h->apmf_len.assign(m->apmf_len, m->apmf_len + rows);
        std::vector<int> aoff(rows + 1, 0);
        for (size_t r = 0; r < rows; r++) {
            if (h->apmf_len[r] < 1) return fail_create(h, SDPB_ERR_ARG, "empty action-dependent pmf row");
            aoff[r + 1] = aoff[r] + h->apmf_len[r];
        }
        std::vector<double> ap(m->apmf_p, m->apmf_p + aoff[rows]);
        std::vector<double> ml(m->min_level_t, m->min_level_t + T);
        UP(h->apmf_len, apmf_len, di) UP(aoff, apmf_off, di) UP(ap, apmf_p, dp) UP(ml, min_level_t, dp)
    }
#undef UP
    mark("tables uploaded");

    h->dV.assign(T, nullptr);
    h->dQ.assign(T, nullptr);
    h->dMask.assign(T, nullptr);
    h->solved.assign(T, 0);

    // ---- exact folding of lead-time states (opt-in) ----
    if (h->opt.dedup && m->lead_time >= 1) h->dedup = true;
    if (h->opt.kernel == SDPB_KERNEL_LEAD_Q2 &&
        !(m->cost_kind == SDPB_COST_BACKORDER && m->lead_time == 2 && !h->dedup))
        return fail_create(h, SDPB_ERR_ARG, "SDPB_KERNEL_LEAD_Q2 needs a backorder model with lead_time 2 and dedup off");
    const bool want_vt = !h->dedup && m->cost_kind == SDPB_COST_BACKORDER && m->lead_time == 2 &&
                         (h->opt.kernel == SDPB_KERNEL_AUTO || h->opt.kernel == SDPB_KERNEL_LEAD_Q2);

    // ---- which part of every V_t this handle holds ----
    // Unsharded: everything.  Sharded: the rows the shard's kernels read (sdpb_shard_reads) plus a guard margin of
    // kWindowMarginRows inventory rows on either side -- register-window kernels prefetch a few levels past the
    // last one they use -- clipped to the grid; the whole (padded) table when that is most of it anyway, so
    // that an in-place all-gather stays possible.
    constexpr long long kWindowMarginRows = 16;
    h->vlo = 0;
    h->vhi = h->Spad;
    if (h->opt.shard_count > 1) {
        int64_t rlo = 0, rhi = S;
        sdpb_shard_reads(h, &rlo, &rhi);
        const long long per_x = S / d.nI;
        const long long wlo = std::max<long long>(0, rlo - kWindowMarginRows * per_x);
        const long long whi = std::min<long long>(S, rhi + kWindowMarginRows * per_x);
        if (rhi > rlo && (double)(whi - wlo) < 0.8 * (double)S) { h->vlo = wlo; h->vhi = whi; }
        if (rhi <= rlo) { h->vlo = 0; h->vhi = 0; }  // an empty shard (more ranks than states) holds nothing
    }
    const long long vlen = h->vhi - h->vlo, qlen = h->hi - h->lo;
    // tables start on 256-byte boundaries and keep the alignment absolute index i would have in a full table:
    // element vlo sits (vlo % 32) doubles into its slot, so address(V[i]) == 8 * i (mod 256)
    auto round256 = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t v_pad = (size_t)(h->vlo % 32) * sizeof(double), q_pad = (size_t)(h->lo % 64) * sizeof(int);
    const size_t v_slot = round256(v_pad + (size_t)vlen * sizeof(double) + 256);
    const size_t q_slot = round256(q_pad + (size_t)qlen * sizeof(int) + 256);
    const int n_vtabs = T + (want_vt ? 1 : 0) + (m->terminal_value ? 1 : 0);
    char* vbase = nullptr;
    char* qbase = nullptr;
    if (h->opt.shard_count > 1) {
        // one plain cudaMalloc allocation: [header: peer flags][V tables][Q tables]
        const size_t need = kSlabHeader + (size_t)n_vtabs * v_slot + (size_t)T * q_slot;
        h->slab = slab_acquire(dev, need, &h->slab_bytes);
        if (!h->slab) return fail_create(h, SDPB_ERR_NOMEM, "allocation of the shard's tables failed");
        h->device_bytes += need;
        if (cudaMemsetAsync(h->slab, 0, kSlabHeader, h->stream) != cudaSuccess)
            return fail_create(h, SDPB_ERR_CUDA, "cudaMemset of the peer flags failed");
        vbase = h->slab + kSlabHeader;
        qbase = vbase + (size_t)n_vtabs * v_slot;
    } else {
        void* p = nullptr;
        if (dev_alloc(h, &p, (size_t)n_vtabs * v_slot) != cudaSuccess)
            return fail_create(h, SDPB_ERR_NOMEM, "allocation of the value tables failed");
        vbase = (char*)p;
        if (dev_alloc(h, &p, (size_t)T * q_slot) != cudaSuccess)
            return fail_create(h, SDPB_ERR_NOMEM, "allocation of the policy tables failed");
        qbase = (char*)p;
    }
    h->v_off0 = (size_t)(vbase - (h->slab ? h->slab : vbase)) + v_pad;
    h->v_stride = v_slot;
    auto v_table = [&](int k) { return reinterpret_cast<double*>(vbase + (size_t)k * v_slot + v_pad) - h->vlo; };
    for (int t = 0; t < T; t++) {
        h->dV[t] = v_table(t);
        h->dQ[t] = reinterpret_cast<int*>(qbase + (size_t)t * q_slot + q_pad) - h->lo;
    }
    int next_tab = T;
    if (want_vt) h->dVT = v_table(next_tab++);  // transposed successor table for the lead-time-2 kernel
    if (m->terminal_value) {
        h->dTerm = v_table(next_tab++);
        if (vlen > 0 && cudaMemcpyAsync(h->dTerm + h->vlo, m->terminal_value + h->vlo,
                                        (size_t)(std::min<long long>(h->vhi, S) - h->vlo) * sizeof(double),
                                        cudaMemcpyHostToDevice, h->stream) != cudaSuccess)
            return fail_create(h, SDPB_ERR_CUDA, "upload of the terminal value table failed");
        // pageable host memory: the copy has left the caller's buffer when the call returns; make it so for
        // page-locked buffers too (the caller owns terminal_value only until sdpb_create returns)
        if (cudaStreamSynchronize(h->stream) != cudaSuccess)
            return fail_create(h, SDPB_ERR_CUDA, "upload of the terminal value table failed");
        // (h->m.terminal_value keeps the caller's pointer value as a marker only; it is never dereferenced again)
    }
    {
        void* p = nullptr;
        if (dev_alloc(h, &p, 4 * sizeof(unsigned long long)) != cudaSuccess)
            return fail_create(h, SDPB_ERR_NOMEM, "allocation failed");
        h->dCounters = (unsigned long long*)p;
    }
    mark("V/Q allocated");
    if (h->dedup) {
        h->vS = (long long)(d.nI + d.nQ - 1) * (m->lead_time >= 2 ? d.nQ : 1) * d.nW;
        void* p = nullptr;
        if (dev_alloc(h, &p, (size_t)h->vS * sizeof(double)) != cudaSuccess)
            return fail_create(h, SDPB_ERR_NOMEM, "allocation of the folded value table failed");
        h->dHv = (double*)p;
        if (dev_alloc(h, &p, (size_t)h->vS * sizeof(int)) != cudaSuccess)
            return fail_create(h, SDPB_ERR_NOMEM, "allocation of the folded policy table failed");
        h->dHa = (int*)p;
    }

    // ---- kernel plan ----
    plan_tiled(h->tiled, h->m, h->dm, h->pmf_len, h->pmf_off, pdi, h->opt.dedup != 0, sm_count);
    plan_cash(h->cash, h->m, h->dm, h->pmf_len, h->pmf_off, pdi);
    h->tiled.variant = h->opt.kernel == SDPB_KERNEL_TILED2 ? 2 : (h->opt.kernel == SDPB_KERNEL_TILED ? 1 : 0);
    if ((h->opt.kernel == SDPB_KERNEL_TILED || h->opt.kernel == SDPB_KERNEL_TILED2) && !h->tiled.available &&
        !(m->cost_kind == SDPB_COST_BACKORDER && m->lead_time >= 1) && !h->cash.available)
        return fail_create(h, SDPB_ERR_ARG, std::string("no shared-memory kernel for this model: ") + h->tiled.why_not);
    h->sm_count = sm_count;
    if (h->opt.kernel == SDPB_KERNEL_AUTO || h->opt.kernel == SDPB_KERNEL_FUSED) {
        plan_fused(h->fused, h->m, h->dm, h->pmf_len, h->pmf_off, pdi, sm_count, h->opt.shard_count);
        // AUTO: the fused kernel trades arithmetic efficiency (5 fp64 instructions per evaluation, one CTA per SM)
        // for having no per-period launch, window-merge or action-split overhead; measured against the tiled
        // path (tools/time_small_grids.py) it wins on grids of up to ~1500 states and on short action lists
        if (h->opt.kernel == SDPB_KERNEL_AUTO &&
            !(h->S <= 1500 || (double)h->S * (m->max_order_idx + 1) <= 1.1e5))
            h->fused.ok = false;
        if (h->fused.ok) {
            std::vector<int> off(h->pmf_off.begin(), h->pmf_off.begin() + T);
            if (upload(h, h->pmf_len, &h->fused.d_len) != SDPB_OK || upload(h, off, &h->fused.d_off) != SDPB_OK ||
                upload(h, h->fused.dimax, &h->fused.d_dimax) != SDPB_OK ||
                upload(h, h->dV, &h->fused.d_V) != SDPB_OK || upload(h, h->dQ, &h->fused.d_Q) != SDPB_OK)
                return fail_create(h, SDPB_ERR_NOMEM, "allocation of the fused-solve tables failed");
        }
    }
    if (h->opt.kernel == SDPB_KERNEL_FUSED && !h->fused.ok)
        return fail_create(h, SDPB_ERR_ARG, "SDPB_KERNEL_FUSED needs an unsharded lead-0 backorder model with the "
                                            "inventory clamp, no G(y) pass and at most 64 states per SM");
    if (h->opt.kernel == SDPB_KERNEL_COLLAPSED) {
        if (!collapsed_ok(h->m) || h->opt.shard_count != 1 || h->dedup)
            return fail_create(h, SDPB_ERR_ARG, "SDPB_KERNEL_COLLAPSED needs an unsharded lead-0 backorder model with the "
                                                "inventory clamp, no G(y) pass and no SDPB_F_NO_ORDER_LAST");
        void* p = nullptr;
        if (dev_alloc(h, &p, ((size_t)h->dm.nI + h->m.max_order_idx + 1) * sizeof(double)) != cudaSuccess)
            return fail_create(h, SDPB_ERR_NOMEM, "allocation of the level table failed");
        h->dG = (double*)p;
        int dmin = 0, dmax = 0;
        bool long_pmf = false;
        for (int v : h->pmf_di) { dmin = std::min(dmin, v); dmax = std::max(dmax, v); }
        for (int len : h->pmf_len) long_pmf = long_pmf || len > 2000;
        if (long_pmf) return fail_create(h, SDPB_ERR_ARG, "SDPB_KERNEL_COLLAPSED: demand support too long");
        h->lc_il0 = -(long long)dmax;
        const long long n_lc = (long long)h->dm.nI + h->m.max_order_idx - dmin + dmax + 1;
        if (dev_alloc(h, &p, (size_t)n_lc * sizeof(double)) != cudaSuccess)
            return fail_create(h, SDPB_ERR_NOMEM, "allocation of the level-cost table failed");
        h->dLc = (double*)p;
        collapsed_level_costs<<<(unsigned)((n_lc + 255) / 256), 256, 0, h->stream>>>(h->dm, h->lc_il0, n_lc, h->dLc);
        if (cudaGetLastError() != cudaSuccess) return fail_create(h, SDPB_ERR_CUDA, "level-cost kernel launch failed");
    }
    h->period_kernel.resize(T);
    for (int t = 1; t <= T; t++) h->period_kernel[t - 1] = choose_period_kernel(h, t);
    mark("planned");
    *out = h;
    return SDPB_OK;
}

int sdpb_shard_reads(const sdpb_handle* h, int64_t* lo, int64_t* hi) {
    if (!h || !lo || !hi) return SDPB_ERR_ARG;
    const DevModel& d = h->dm;
    const sdpb_model& m = h->m;
    *lo = 0;
    *hi = h->S;
    if (h->hi <= h->lo) { *hi = 0; return SDPB_OK; }
    // folded solves walk the whole virtual grid on every rank; the workforce kind can lose every employee
    if (h->dedup || staff_kind(m)) return SDPB_OK;
    const long long per_x = h->S / d.nI;  // the first inventory axis is outermost
    long long r0 = h->lo / per_x, r1 = (h->hi - 1) / per_x;
    int dmin = 0, dmax = 0;
    for (int v : h->pmf_di) { dmin = std::min(dmin, v); dmax = std::max(dmax, v); }
    // successor level = x + (order or pipeline quantity, at most max_order_idx) - demand, then clamps
    r0 -= dmax;
    r1 += (long long)m.max_order_idx - dmin;
    if (m.flags & SDPB_F_LOST_SALES) {  // levels below zero are lifted to the zero row
        r0 = std::min<long long>(r0, d.i_zero);
        r1 = std::max<long long>(r1, d.i_zero);
    }
    r0 = std::max<long long>(r0, 0);
    r1 = std::min<long long>(r1, d.nI - 1);
    *lo = r0 * per_x;
    *hi = (r1 + 1) * per_x;
    return SDPB_OK;
}

int sdpb_grid_info(const sdpb_handle* h, sdpb_grid* g) {
    if (!h || !g) return SDPB_ERR_ARG;
    g->ndim = h->ndim;
    g->n_inv = h->dm.nI;
    g->n_cash = h->dm.nW;
    g->n_q = h->dm.nQ;
    g->n_states = h->S;
    g->shard_lo = h->lo;
    g->shard_hi = h->hi;
    g->n_actions = h->m.max_order_idx + 1;
    g->T = h->m.T;
    g->cash_k_min = h->dm.kmin;
    g->window_lo = h->vlo;
    g->window_hi = h->vhi;
    g->device_bytes = (int64_t)h->device_bytes;
    return SDPB_OK;
}

int sdpb_solve_period_async(sdpb_handle* h, int period) {
    if (!h) return SDPB_ERR_ARG;
    CU(cudaSetDevice(h->device));
    return solve_period(h, period);
}

int sdpb_sync(sdpb_handle* h) {
    if (!h) return SDPB_ERR_ARG;
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    if (h->peer.attached) return finish_sharded(h);  // did a peer fail to deliver?
    return SDPB_OK;
}

// The whole horizon in one cooperative launch (kernel_fused.cuh).  SDPB_ERR_STATE: not launched, use the
// per-period path.
static int enqueue_fused(sdpb_handle* h) {
    FusedPlan& P = h->fused;
    FusedArgs a;
    a.T = h->m.T; a.A = h->m.max_order_idx + 1; a.BX = P.BX; a.WN = P.WN; a.Dmax = P.Dmax;
    a.len = P.d_len; a.off = P.d_off; a.di_max = P.d_dimax; a.V = P.d_V; a.Q = P.d_Q;
    void* fn = h->dm.is_min ? (void*)bi_inv_fused<true> : (void*)bi_inv_fused<false>;
    if (P.smem > 48 * 1024 &&
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.smem) != cudaSuccess) {
        cudaGetLastError();
        return SDPB_ERR_STATE;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kFusedThreads, P.smem) != cudaSuccess ||
        (long long)per_sm * h->sm_count < P.grid) {
        cudaGetLastError();
        return SDPB_ERR_STATE;  // the grid barrier needs every CTA resident
    }
    void* args[] = {(void*)&h->dm, (void*)&a};
    if (cudaLaunchCooperativeKernel(fn, dim3((unsigned)P.grid), dim3(kFusedThreads), args, P.smem, h->stream) != cudaSuccess) {
        cudaGetLastError();
        return SDPB_ERR_STATE;
    }
    std::fill(h->solved.begin(), h->solved.end(), 1);
    h->stats.launches = 1;
    h->stats.kernel_used = SDPB_KERNEL_FUSED;
    for (int t = 1; t <= h->m.T; t++) {
        const double ev = count_evals_period(h, t);
        h->stats.evals += ev;
        h->stats.evals_executed += ev;
        h->stats.fp64_ops += ev * (t == h->m.T ? 3.0 : 5.0);
    }
    return SDPB_OK;
}

static int enqueue_all_periods(sdpb_handle* h) {
    std::fill(h->solved.begin(), h->solved.end(), 0);
    h->stats = sdpb_stats{};
    // (one of a wide batch: the whole-horizon kernel is a cooperative launch sized for the whole GPU, and a batch of
    //  them would run one after the other; the per-period kernels of different instances run side by side)
    const bool in_wide_batch = h->tiled.batch >= 8 && h->opt.kernel != SDPB_KERNEL_FUSED;
    if (h->fused.ok && !in_wide_batch) {
        const int rc = enqueue_fused(h);
        if (rc != SDPB_ERR_STATE) return rc;
        h->fused.ok = false;  // cannot be launched cooperatively here: per-period launches from now on
    }
    for (int t = h->m.T; t >= 1; t--) {
        int rc = solve_period(h, t);
        if (rc != SDPB_OK) return rc;
    }
    return SDPB_OK;
}

int sdpb_solve_async(sdpb_handle* h) {
    if (!h) return SDPB_ERR_ARG;
    if (h->opt.shard_count != 1) {
        if (!h->peer.attached) {
            h->err = "a sharded handle solves with its peers: connect them first (sdpb_peer_export / sdpb_peer_attach, or "
                     "sdpb_group_create), or step it with sdpb_solve_period_async and exchange V_t yourself";
            return SDPB_ERR_STATE;
        }
        if (h->peer.by_events) {
            h->err = "the shards of one process are solved together: sdpb_group_solve";
            return SDPB_ERR_STATE;
        }
        CU(cudaSetDevice(h->device));
        std::fill(h->solved.begin(), h->solved.end(), 0);
        h->stats = sdpb_stats{};
        for (int t = h->m.T; t >= 1; t--) {
            const int rc = enqueue_period_sharded(h, t, true);
            if (rc != SDPB_OK) return rc;
        }
        h->solve_count++;
        return SDPB_OK;
    }
    CU(cudaSetDevice(h->device));
    h->reached = false;
    if (h->graph_exec) {
        h->stats = h->graph_stats;
        CU(cudaGraphLaunch(h->graph_exec, h->stream));
        return SDPB_OK;
    }
    if (h->solve_count >= 1 && !h->graph_failed && !h->fused.ok) {  // (a fused solve is one launch already)
        // second solve: every scratch buffer exists by now, so the launches can be captured
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            int rc = enqueue_all_periods(h);
            cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
            if (rc == SDPB_OK && e == cudaSuccess && graph &&
                cudaGraphInstantiate(&h->graph_exec, graph, 0) == cudaSuccess) {
                cudaGraphDestroy(graph);
                h->graph_stats = h->stats;
                CU(cudaGraphLaunch(h->graph_exec, h->stream));
                h->solve_count++;
                return SDPB_OK;
            }
            if (graph) cudaGraphDestroy(graph);
            h->graph_exec = nullptr;
        }
        cudaGetLastError();
        h->graph_failed = true;  // fall back to plain launches for good
    }
    int rc = enqueue_all_periods(h);
    if (rc == SDPB_OK) h->solve_count++;
    return rc;
}

int sdpb_solve(sdpb_handle* h) {
    if (!h) return SDPB_ERR_ARG;
    CU(cudaSetDevice(h->device));
    CU(cudaEventRecord(h->ev0, h->stream));
    int rc = sdpb_solve_async(h);
    if (rc != SDPB_OK) return rc;
    CU(cudaEventRecord(h->ev1, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->stats.solve_ms = ms;
    h->stats.kernel_ms = ms;
    if (h->opt.shard_count != 1) return finish_sharded(h);
    return SDPB_OK;
}

int sdpb_value(sdpb_handle* h, int period, const double* states, int n, double* v, double* q) {
    if (!h || !states || n < 0) return SDPB_ERR_ARG;
    if (period < 1 || period > h->m.T) { h->err = "period out of range"; return SDPB_ERR_ARG; }
    if (!h->solved[period - 1]) { h->err = "period not solved"; return SDPB_ERR_STATE; }
    if (n == 0) return SDPB_OK;
    CU(cudaSetDevice(h->device));
    std::vector<long long> idx(n);
    for (int i = 0; i < n; i++) {
        idx[i] = index_of_state(h, states + (size_t)i * h->ndim);
        if (idx[i] < 0) {
            h->err = "state " + std::to_string(i) + " is not a grid point (the reference would throw a "
                     "NullPointerException from getAction on an unsolved state)";
            return SDPB_ERR_UNSOLVED;
        }
        if (h->opt.shard_count > 1 && (idx[i] < h->lo || idx[i] >= h->hi)) {
            h->err = "state " + std::to_string(i) + " is owned by another shard (sdpb_group_value routes queries)";
            return SDPB_ERR_UNSOLVED;
        }
    }
    long long* dIdx = nullptr;
    double* dv = nullptr;
    int* dq = nullptr;
    // scratch from the stream-ordered pool: plain cudaMalloc/cudaFree synchronise the device and cost
    // tens of milliseconds next to large pooled tables
    CU(pool_alloc(h, (void**)&dIdx, n * sizeof(long long)));
    CU(pool_alloc(h, (void**)&dv, n * sizeof(double)));
    CU(pool_alloc(h, (void**)&dq, n * sizeof(int)));
    std::vector<double> hv(n);
    std::vector<int> hq(n);
    cudaError_t e = cudaMemcpyAsync(dIdx, idx.data(), n * sizeof(long long), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) {
        gather_vq<<<(n + 255) / 256, 256, 0, h->stream>>>(dIdx, n, h->dV[period - 1], h->dQ[period - 1], dv, dq);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(hv.data(), dv, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hq.data(), dq, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    cudaFreeAsync(dIdx, h->stream); cudaFreeAsync(dv, h->stream); cudaFreeAsync(dq, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { h->err = std::string("sdpb_value: ") + cudaGetErrorString(e); return SDPB_ERR_CUDA; }
    for (int i = 0; i < n; i++) {
        if (v) v[i] = hv[i];
        if (q) q[i] = q_of_index(h, idx[i], hq[i]);
    }
    return SDPB_OK;
}

// V_t / Q_t of the flattened range [a, b) (inside what the handle holds) into host buffers that start at `a`.
static int copy_tables(sdpb_handle* h, int period, long long a, long long b, double* V, double* Q) {
    CU(cudaSetDevice(h->device));
    const long long n = b - a;
    if (n <= 0) return SDPB_OK;
    if (V) CU(cudaMemcpyAsync(V, h->dV[period - 1] + a, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (!Q) CU(cudaStreamSynchronize(h->stream));
    if (Q) {
        double* dq = nullptr;
        CU(pool_alloc(h, (void**)&dq, (size_t)n * sizeof(double)));
        policy_to_double<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(
            h->dQ[period - 1] + a, dq, n, h->m.step, h->m.cost_kind == SDPB_COST_CASH_XR, h->m.inv_min,
            (long long)h->dm.nW, a);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(Q, dq, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
        cudaFreeAsync(dq, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) { h->err = std::string("sdpb_period_tables: ") + cudaGetErrorString(e); return SDPB_ERR_CUDA; }
    }
    return SDPB_OK;
}

int sdpb_period_tables(sdpb_handle* h, int period, double* V, double* Q) {
    if (!h) return SDPB_ERR_ARG;
    if (period < 1 || period > h->m.T) { h->err = "period out of range"; return SDPB_ERR_ARG; }
    if (!h->solved[period - 1]) { h->err = "period not solved"; return SDPB_ERR_STATE; }
    // a sharded handle fills its own block of the caller's n_states-long buffers and leaves the rest alone
    return copy_tables(h, period, h->lo, h->hi, V ? V + h->lo : nullptr, Q ? Q + h->lo : nullptr);
}

int sdpb_shard_tables(sdpb_handle* h, int period, double* V, double* Q) {
    if (!h) return SDPB_ERR_ARG;
    if (period < 1 || period > h->m.T) { h->err = "period out of range"; return SDPB_ERR_ARG; }
    if (!h->solved[period - 1]) { h->err = "period not solved"; return SDPB_ERR_STATE; }
    return copy_tables(h, period, h->lo, h->hi, V, Q);
}

int sdpb_device_tables(sdpb_handle* h, int period, void** dV, void** dQidx) {
    if (!h) return SDPB_ERR_ARG;
    if (period < 1 || period > h->m.T) { h->err = "period out of range"; return SDPB_ERR_ARG; }
    // first element held: V_t[window_lo] and Q_t[shard_lo] (sdpb_grid_info); the whole table when unsharded
    if (dV) *dV = h->dV[period - 1] + h->vlo;
    if (dQidx) *dQidx = h->dQ[period - 1] + h->lo;
    return SDPB_OK;
}

int sdpb_state_of_index(const sdpb_handle* h, int64_t idx, double* state) {
    if (!h || !state || idx < 0 || idx >= h->S) return SDPB_ERR_ARG;
    state_of_index(h, idx, state, nullptr);
    return SDPB_OK;
}

int sdpb_reach(sdpb_handle* h, const double* init_states, int n) {
    if (!h || !init_states || n < 1) return SDPB_ERR_ARG;
    if (h->opt.shard_count != 1) { h->err = "sdpb_reach needs an unsharded handle"; return SDPB_ERR_STATE; }

    CU(cudaSetDevice(h->device));
    const int T = h->m.T;
    for (int t = 0; t < T; t++) {
        if (!h->dMask[t]) {
            void* p = nullptr;
            CU(dev_alloc(h, &p, (size_t)h->S));
            h->dMask[t] = (unsigned char*)p;
        }
        CU(cudaMemsetAsync(h->dMask[t], 0, (size_t)h->S, h->stream));
    }
    for (int i = 0; i < n; i++) {
        long long idx = index_of_state(h, init_states + (size_t)i * h->ndim);
        if (idx < 0) { h->err = "initial state is not a grid point"; return SDPB_ERR_UNSOLVED; }
        CU(cudaMemsetAsync(h->dMask[0] + idx, 1, 1, h->stream));
    }
    const bool surv = h->m.recursion == SDPB_REC_SURVIVAL;
    CU(cudaMemsetAsync(h->dCounters, 0, 4 * sizeof(unsigned long long), h->stream));
    // periods 1..T-1 mark their successors; period T is visited only to see whether a reached state's action
    // set was capped (mask_n == nullptr: no transition is evaluated)
    for (int t = 1; t <= T; t++) {
        switch (h->m.cost_kind) {
        case SDPB_COST_BACKORDER: launch_reach<SDPB_COST_BACKORDER, false>(h, t); break;
        case SDPB_COST_CASH_DEPOSIT:
            if (surv) launch_reach<SDPB_COST_CASH_DEPOSIT, true>(h, t);
            else launch_reach<SDPB_COST_CASH_DEPOSIT, false>(h, t);
            break;
        case SDPB_COST_CASH_OVERDRAFT:
            if (surv) launch_reach<SDPB_COST_CASH_OVERDRAFT, true>(h, t);
            else launch_reach<SDPB_COST_CASH_OVERDRAFT, false>(h, t);
            break;
        case SDPB_COST_CASH_XR: launch_reach<SDPB_COST_CASH_XR, false>(h, t); break;
        case SDPB_COST_CASH_OD_LIMIT: launch_reach<SDPB_COST_CASH_OD_LIMIT, false>(h, t); break;
        case SDPB_COST_CASH_OD_TESTING: launch_reach<SDPB_COST_CASH_OD_TESTING, false>(h, t); break;
        case SDPB_COST_CASH_LOAN: launch_reach<SDPB_COST_CASH_LOAN, false>(h, t); break;
        case SDPB_COST_CASH_TWO_PRODUCT:
            if (t < T)
                reach_two_product<<<(unsigned)((h->S + 127) / 128), 128, 0, h->stream>>>(
                    h->dm, t, h->pmf_len[t - 1], h->pmf_off[t - 1], h->dMask[t - 1], h->dMask[t], h->dCounters);
            break;
        case SDPB_COST_STAFF:
            if (t < T)
                reach_staff<<<(unsigned)((h->S + 127) / 128), 128, 0, h->stream>>>(h->dm, t, h->dMask[t - 1], h->dMask[t]);
            break;
        }
        CU(cudaGetLastError());
    }
    unsigned long long cnt[4] = {0, 0, 0, 0};
    CU(cudaMemcpyAsync(cnt, h->dCounters, sizeof cnt, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->reached = true;
    for (int k = 0; k < 3; k++) h->reach_cnt[k] = (double)cnt[k];  // reported by sdpb_stats_get
    // A dense-grid artefact at a state the reference itself would visit changes that state's value: refuse unless
    // the caller said it is acceptable.  (The mask and the opt table stay available either way.)
    if (cnt[0] && !(h->opt.allow & SDPB_ALLOW_CLIPPED_SUCCESSORS)) {
        h->err = std::to_string(cnt[0]) + " successor(s) of states the reference would visit lie outside the inventory grid of "
                 "a model that does not clamp (they were folded onto the boundary row): enlarge [inv_min, inv_max] "
                 "(sdpb_reachable_hull) or pass SDPB_ALLOW_CLIPPED_SUCCESSORS";
        return SDPB_ERR_OFFGRID;
    }
    if (cnt[1] && !(h->opt.allow & SDPB_ALLOW_CAPPED_ACTIONS)) {
        h->err = std::to_string(cnt[1]) + " reached state(s) have an order-up-to range longer than max_order_idx + 1 "
                 "(CashConstraintXR.java:71-75 has no cap): raise max_order_idx or pass SDPB_ALLOW_CAPPED_ACTIONS";
        return SDPB_ERR_OFFGRID;
    }
    if (cnt[2] && h->opt.strict_cash_bounds) {
        h->err = std::to_string(cnt[2]) + " successor(s) of reached states had their cash clamped at cash_min / cash_max "
                 "(strict_cash_bounds)";
        return SDPB_ERR_OFFGRID;
    }
    return SDPB_OK;
}

int sdpb_opt_table(sdpb_handle* h, double* rows, size_t* nrows) {
    if (!h || !nrows) return SDPB_ERR_ARG;
    if (!h->reached) { h->err = "call sdpb_reach first"; return SDPB_ERR_STATE; }
    for (int t = 0; t < h->m.T; t++)
        if (!h->solved[t]) { h->err = "not solved"; return SDPB_ERR_STATE; }
    CU(cudaSetDevice(h->device));
    const size_t cap = *nrows;
    const int w = h->ndim + 2;
    size_t count = 0;
    std::vector<unsigned char> mask((size_t)h->S);
    std::vector<int> hq;
    if (rows) hq.resize((size_t)h->S);
    for (int t = 0; t < h->m.T; t++) {
        CU(cudaMemcpy(mask.data(), h->dMask[t], (size_t)h->S, cudaMemcpyDeviceToHost));
        if (rows) CU(cudaMemcpy(hq.data(), h->dQ[t], (size_t)h->S * sizeof(int), cudaMemcpyDeviceToHost));
        for (long long i = 0; i < h->S; i++) {
            if (!mask[i]) continue;
            if (rows && count < cap) {
                double* r = rows + count * w;
                r[0] = t + 1;
                state_of_index(h, i, r + 1, nullptr);
                r[w - 1] = q_of_index(h, i, hq[i]);
            }
            count++;
        }
    }
    *nrows = count;
    return SDPB_OK;
}

int sdpb_eval_triples(sdpb_handle* h, int period, const double* states, const int32_t* action_idx,
                      const double* demand, int n, double* c, double* next_states, int32_t* n_actions) {
    if (!h || !states || !action_idx || !demand || n < 1) return SDPB_ERR_ARG;
    if (period < 1 || period > h->m.T) { h->err = "period out of range"; return SDPB_ERR_ARG; }
    if (two_product(h->m) || staff_kind(h->m)) { h->err = "sdpb_eval_triples is not implemented for two-product and staff models"; return SDPB_ERR_ARG; }
    CU(cudaSetDevice(h->device));
    std::vector<long long> sidx(n), hnext(n);
    std::vector<int> demi(n), hna(n);
    std::vector<double> hc(n);
    for (int i = 0; i < n; i++) {
        sidx[i] = index_of_state(h, states + (size_t)i * h->ndim);
        if (sidx[i] < 0) { h->err = "state is not a grid point"; return SDPB_ERR_UNSOLVED; }
        double f = demand[i] / h->m.step;
        if (!is_int(f)) { h->err = "demand is not a multiple of step"; return SDPB_ERR_OFFGRID; }
        demi[i] = (int)f;
        if (action_idx[i] < 0 || action_idx[i] > h->m.max_order_idx) { h->err = "action index out of range"; return SDPB_ERR_ARG; }
    }
    long long *dS = nullptr, *dN = nullptr;
    int *dA = nullptr, *dDi = nullptr, *dNa = nullptr;
    double *dD = nullptr, *dC = nullptr;
    cudaError_t e = cudaSuccess;
    auto al = [&](void** p, size_t b) { if (e == cudaSuccess) e = pool_alloc(h, p, b); };
    al((void**)&dS, n * 8); al((void**)&dN, n * 8); al((void**)&dA, n * 4); al((void**)&dDi, n * 4);
    al((void**)&dNa, n * 4); al((void**)&dD, n * 8); al((void**)&dC, n * 8);
    auto cp = [&](void* d, const void* s, size_t b, cudaMemcpyKind k) { if (e == cudaSuccess) e = cudaMemcpyAsync(d, s, b, k, h->stream); };
    cp(dS, sidx.data(), n * 8, cudaMemcpyHostToDevice);
    cp(dA, action_idx, n * 4, cudaMemcpyHostToDevice);
    cp(dDi, demi.data(), n * 4, cudaMemcpyHostToDevice);
    cp(dD, demand, n * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        const int blocks = (n + 127) / 128;
        switch (h->m.cost_kind) {
        case SDPB_COST_BACKORDER: eval_triples<SDPB_COST_BACKORDER><<<blocks, 128, 0, h->stream>>>(h->dm, period, n, dS, dA, dD, dDi, dC, dN, dNa); break;
        case SDPB_COST_CASH_DEPOSIT: eval_triples<SDPB_COST_CASH_DEPOSIT><<<blocks, 128, 0, h->stream>>>(h->dm, period, n, dS, dA, dD, dDi, dC, dN, dNa); break;
        case SDPB_COST_CASH_OVERDRAFT: eval_triples<SDPB_COST_CASH_OVERDRAFT><<<blocks, 128, 0, h->stream>>>(h->dm, period, n, dS, dA, dD, dDi, dC, dN, dNa); break;
        case SDPB_COST_CASH_XR: eval_triples<SDPB_COST_CASH_XR><<<blocks, 128, 0, h->stream>>>(h->dm, period, n, dS, dA, dD, dDi, dC, dN, dNa); break;
        case SDPB_COST_CASH_OD_LIMIT: eval_triples<SDPB_COST_CASH_OD_LIMIT><<<blocks, 128, 0, h->stream>>>(h->dm, period, n, dS, dA, dD, dDi, dC, dN, dNa); break;
        case SDPB_COST_CASH_OD_TESTING: eval_triples<SDPB_COST_CASH_OD_TESTING><<<blocks, 128, 0, h->stream>>>(h->dm, period, n, dS, dA, dD, dDi, dC, dN, dNa); break;
        case SDPB_COST_CASH_LOAN: eval_triples<SDPB_COST_CASH_LOAN><<<blocks, 128, 0, h->stream>>>(h->dm, period, n, dS, dA, dD, dDi, dC, dN, dNa); break;
        }
        e = cudaGetLastError();
    }
    cp(hc.data(), dC, n * 8, cudaMemcpyDeviceToHost);
    cp(hnext.data(), dN, n * 8, cudaMemcpyDeviceToHost);
    cp(hna.data(), dNa, n * 4, cudaMemcpyDeviceToHost);
    for (void* p : {(void*)dS, (void*)dN, (void*)dA, (void*)dDi, (void*)dNa, (void*)dD, (void*)dC})
        if (p) cudaFreeAsync(p, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { h->err = std::string("sdpb_eval_triples: ") + cudaGetErrorString(e); return SDPB_ERR_CUDA; }
    for (int i = 0; i < n; i++) {
        if (c) c[i] = hc[i];
        if (next_states) state_of_index(h, hnext[i], next_states + (size_t)i * h->ndim, nullptr);
        if (n_actions) n_actions[i] = hna[i];
    }
    return SDPB_OK;
}

int sdpb_simulate(sdpb_handle* h, const double* init_state, const double* samples, int n, double discount,
                  double* values) {
    if (!h || !init_state || !samples || !values || n < 1) return SDPB_ERR_ARG;
    if (h->opt.shard_count != 1) { h->err = "sdpb_simulate needs an unsharded handle"; return SDPB_ERR_STATE; }
    if (two_product(h->m) || staff_kind(h->m)) { h->err = "sdpb_simulate is not implemented for two-product and staff models"; return SDPB_ERR_ARG; }
    const int T = h->m.T;
    for (int t = 0; t < T; t++)
        if (!h->solved[t]) { h->err = "not solved"; return SDPB_ERR_STATE; }
    const long long init_idx = index_of_state(h, init_state);
    if (init_idx < 0) { h->err = "initial state is not a grid point"; return SDPB_ERR_UNSOLVED; }
    CU(cudaSetDevice(h->device));
    std::vector<double> pw(T);
    for (int t = 0; t < T; t++) pw[t] = std::pow(discount, (double)t);  // Math.pow(discountFactor, t)
    std::vector<const int*> qptr(h->dQ.begin(), h->dQ.end());
    double *dS = nullptr, *dP = nullptr, *dV = nullptr;
    const int** dQp = nullptr;
    int* dOff = nullptr;
    cudaError_t e = cudaSuccess;
    auto al = [&](void** p, size_t b) { if (e == cudaSuccess) e = pool_alloc(h, p, b); };
    al((void**)&dS, (size_t)n * T * 8); al((void**)&dP, (size_t)T * 8); al((void**)&dV, (size_t)n * 8);
    al((void**)&dQp, (size_t)T * sizeof(int*)); al((void**)&dOff, 4);
    auto cp = [&](void* d, const void* s, size_t b, cudaMemcpyKind k) { if (e == cudaSuccess) e = cudaMemcpyAsync(d, s, b, k, h->stream); };
    cp(dS, samples, (size_t)n * T * 8, cudaMemcpyHostToDevice);
    cp(dP, pw.data(), (size_t)T * 8, cudaMemcpyHostToDevice);
    cp(dQp, qptr.data(), (size_t)T * sizeof(int*), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemsetAsync(dOff, 0, 4, h->stream);
    int off = 0;
    if (e == cudaSuccess) {
        const int blocks = (n + 127) / 128;
#define SDPB_SIM(K) case K: simulate_paths<K><<<blocks, 128, 0, h->stream>>>(h->dm, init_idx, dS, n, dP, dQp, dV, dOff); break;
        switch (h->m.cost_kind) {
            SDPB_SIM(SDPB_COST_BACKORDER) SDPB_SIM(SDPB_COST_CASH_DEPOSIT) SDPB_SIM(SDPB_COST_CASH_OVERDRAFT)
            SDPB_SIM(SDPB_COST_CASH_XR) SDPB_SIM(SDPB_COST_CASH_OD_LIMIT) SDPB_SIM(SDPB_COST_CASH_OD_TESTING)
            SDPB_SIM(SDPB_COST_CASH_LOAN)
        }
#undef SDPB_SIM
        e = cudaGetLastError();
    }
    cp(values, dV, (size_t)n * 8, cudaMemcpyDeviceToHost);
    cp(&off, dOff, 4, cudaMemcpyDeviceToHost);
    for (void* p : {(void*)dS, (void*)dP, (void*)dV, (void*)dQp, (void*)dOff})
        if (p) cudaFreeAsync(p, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { h->err = std::string("sdpb_simulate: ") + cudaGetErrorString(e); return SDPB_ERR_CUDA; }
    if (off) { h->err = "a rounded sample demand is not a multiple of step"; return SDPB_ERR_OFFGRID; }
    return SDPB_OK;
}

int sdpb_microbench(int device, double* nofma_tops, double* fma_tflops, double* lds_gbs) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return SDPB_ERR_NO_DEVICE;
    if (device < 0) cudaGetDevice(&device);
    if (device >= ndev || cudaSetDevice(device) != cudaSuccess) return SDPB_ERR_NO_DEVICE;
    int sm_count = 0;
    if (cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return SDPB_ERR_CUDA;
    const int blocks = sm_count * 8, threads = 256;
    double* out = nullptr;
    if (cudaMalloc(&out, (size_t)blocks * threads * sizeof(double)) != cudaSuccess) return SDPB_ERR_NOMEM;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    auto best_ms = [&](auto launch) {
        float best = 1e30f;
        for (int rep = 0; rep < 6; rep++) {
            cudaEventRecord(e0);
            launch();
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep > 0 && ms < best) best = ms;
        }
        return (double)best;
    };
    const int iters = 20000;
    const double n_thr = (double)blocks * threads;
    double ms = best_ms([&] { mb_fp64_nofma<<<blocks, threads>>>(out, iters, 1.0000001, 1e-7); });
    if (nofma_tops) *nofma_tops = n_thr * iters * kMbChains * 2.0 / (ms * 1e-3) / 1e12;
    ms = best_ms([&] { mb_fp64_fma<<<blocks, threads>>>(out, iters, 1.0000001, 1e-7); });
    if (fma_tflops) *fma_tflops = n_thr * iters * kMbChains * 2.0 * 2.0 / (ms * 1e-3) / 1e12;
    const int lds_iters = 20000;
    ms = best_ms([&] { mb_lds128<<<blocks, threads>>>(out, lds_iters); });
    if (lds_gbs) *lds_gbs = n_thr * lds_iters * 4.0 * 16.0 / (ms * 1e-3) / 1e9;
    cudaError_t e = cudaGetLastError();
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    return e == cudaSuccess ? SDPB_OK : SDPB_ERR_CUDA;
}

// ---- multi-GPU: connecting the shards ------------------------------------------------------------------------------
int sdpb_peer_export(sdpb_handle* h, void* blob) {
    if (!h || !blob) return SDPB_ERR_ARG;
    if (h->opt.shard_count < 2 || !h->slab) { h->err = "sdpb_peer_export needs a sharded handle"; return SDPB_ERR_STATE; }
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));  // the flag words are zero before anybody can see them
    PeerInfo pi;
    std::memset(&pi, 0, sizeof pi);
    pi.magic = kPeerMagic; pi.version = SDPB_ABI_VERSION;
    pi.rank = h->opt.shard_rank; pi.world = h->opt.shard_count; pi.device = h->device; pi.T = h->m.T;
    pi.pid = (int64_t)getpid();
    pi.base = (uint64_t)(uintptr_t)h->slab;
    pi.n_states = h->S; pi.lo = h->lo; pi.hi = h->hi;
    int64_t rlo = 0, rhi = 0;
    sdpb_shard_reads(h, &rlo, &rhi);
    pi.rlo = rlo; pi.rhi = rhi; pi.vlo = h->vlo; pi.vhi = h->vhi;
    pi.v_off0 = h->v_off0; pi.v_stride = h->v_stride; pi.flags_off = 0;
    pi.model_hash = model_hash(h);
    pi.handle = (uint64_t)(uintptr_t)h;
    if (cudaDeviceGetPCIBusId(pi.pci, (int)sizeof pi.pci, h->device) != cudaSuccess) { cudaGetLastError(); pi.pci[0] = 0; }
    CU(cudaIpcGetMemHandle(&pi.ipc, h->slab));
    std::memset(blob, 0, SDPB_PEER_BLOB_BYTES);
    std::memcpy(blob, &pi, sizeof pi);
    return SDPB_OK;
}

int sdpb_peer_attach(sdpb_handle* h, const void* blobs, int n_blobs) {
    if (!h || !blobs) return SDPB_ERR_ARG;
    const int world = h->opt.shard_count, rank = h->opt.shard_rank;
    if (world < 2 || !h->slab) { h->err = "sdpb_peer_attach needs a sharded handle"; return SDPB_ERR_STATE; }
    if (n_blobs != world || world > kMaxPeers) { h->err = "need one blob per shard, in rank order (at most 64 shards)"; return SDPB_ERR_ARG; }
    if (h->peer.attached) { h->err = "already attached"; return SDPB_ERR_STATE; }
    CU(cudaSetDevice(h->device));
    PeerLink& P = h->peer;
    P.info.assign(world, PeerInfo{});
    P.mapped.assign(world, nullptr);
    P.ipc_opened.assign(world, 0);
    const uint64_t my_hash = model_hash(h);
    for (int r = 0; r < world; r++) {
        PeerInfo& pi = P.info[r];
        std::memcpy(&pi, (const char*)blobs + (size_t)r * SDPB_PEER_BLOB_BYTES, sizeof pi);
        if (pi.magic != kPeerMagic || pi.version != SDPB_ABI_VERSION || pi.rank != r || pi.world != world ||
            pi.T != h->m.T || pi.n_states != h->S || pi.model_hash != my_hash) {
            h->err = "blob " + std::to_string(r) + " does not describe shard " + std::to_string(r) + " of this model";
            return SDPB_ERR_ARG;
        }
    }
    // all shards in this process (a group), or every shard in its own process on its own GPU
    int same_pid = 0;
    for (int r = 0; r < world; r++) same_pid += P.info[r].pid == (int64_t)getpid();
    if (same_pid != world && same_pid != 1) { h->err = "shards must either all live in one process or each in its own"; return SDPB_ERR_PEER; }
    P.by_events = same_pid == world;
    if (!P.by_events) {
        // The receivers spin on flag words the senders store: a waiter and the kernel it waits for must never share a
        // GPU (nothing guarantees that two processes' kernels run at the same time; the context switch can time out).
        for (int r = 0; r < world; r++)
            for (int q = r + 1; q < world; q++)
                if (P.info[r].pci[0] && std::strncmp(P.info[r].pci, P.info[q].pci, sizeof P.info[r].pci) == 0) {
                    h->err = "shards " + std::to_string(r) + " and " + std::to_string(q) + " are in different processes on the "
                             "same GPU (" + P.info[r].pci + "): one process per GPU, or all shards in one process (sdpb_group_create)";
                    return SDPB_ERR_PEER;
                }
    } else {
        P.peer_handles.assign(world, nullptr);
        for (int r = 0; r < world; r++) P.peer_handles[r] = reinterpret_cast<sdpb_handle*>((uintptr_t)P.info[r].handle);
        CU(cudaEventCreateWithFlags(&P.ev_pushed, cudaEventDisableTiming));
    }
    for (int r = 0; r < world; r++) {
        const PeerInfo& pi = P.info[r];
        if (r == rank) { P.mapped[r] = h->slab; continue; }
        if (pi.pid == (int64_t)getpid()) {
            // same process (sdpb_group_create): the address is valid as it is; another device needs peer access
            if (pi.device != h->device) {
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, h->device, pi.device) != cudaSuccess || !can) {
                    cudaGetLastError();
                    h->err = "device " + std::to_string(h->device) + " cannot access device " + std::to_string(pi.device) + " (no P2P path)";
                    return SDPB_ERR_PEER;
                }
                const cudaError_t e = cudaDeviceEnablePeerAccess(pi.device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                    h->err = std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e);
                    return SDPB_ERR_PEER;
                }
                cudaGetLastError();
            }
            P.mapped[r] = reinterpret_cast<char*>((uintptr_t)pi.base);
        } else {
            char* p = nullptr;
            const cudaError_t e = ipc_map(pi.ipc, h->device, &p);
            if (e != cudaSuccess) {
                cudaGetLastError();
                h->err = std::string("cudaIpcOpenMemHandle (shard ") + std::to_string(r) + "): " + cudaGetErrorString(e);
                return SDPB_ERR_PEER;
            }
            P.mapped[r] = p;
            P.ipc_opened[r] = 1;
        }
    }
    // who needs which of my rows, and whose rows do I need
    std::vector<unsigned*> targets;
    P.sends.clear(); P.recv_from.clear(); P.bytes_out = P.bytes_in = 0;
    const PeerInfo& me = P.info[rank];
    for (int r = 0; r < world; r++) {
        if (r == rank) continue;
        const PeerInfo& pi = P.info[r];
        const long long a = std::max<long long>(h->lo, pi.rlo), b = std::min<long long>(h->hi, pi.rhi);
        if (b > a) {
            if (a < pi.vlo || b > pi.vhi) { h->err = "a peer's window does not contain the rows it reads"; return SDPB_ERR_PEER; }
            P.sends.push_back({r, a, b});
            targets.push_back(reinterpret_cast<unsigned*>(P.mapped[r] + pi.flags_off) + rank);
            P.bytes_out += (b - a) * 8;
        }
        const long long c = std::max<long long>(pi.lo, me.rlo), d2 = std::min<long long>(pi.hi, me.rhi);
        if (d2 > c) { P.recv_from.push_back(r); P.bytes_in += (d2 - c) * 8; }
    }
    void* p = nullptr;
    {
        std::vector<DevPeer> dp;
        for (const PeerSend& sd : P.sends) {
            const PeerInfo& pi = P.info[sd.rank];
            dp.push_back(DevPeer{P.mapped[sd.rank] + pi.v_off0 - (long long)pi.vlo * (long long)sizeof(double), pi.v_stride, sd.a, sd.b});
        }
        CU(dev_alloc(h, &p, std::max<size_t>(1, dp.size()) * sizeof(DevPeer)));
        P.d_peers = p;
        if (!dp.empty()) CU(cudaMemcpyAsync(P.d_peers, dp.data(), dp.size() * sizeof(DevPeer), cudaMemcpyHostToDevice, h->stream));
    }
    CU(dev_alloc(h, &p, std::max<size_t>(1, targets.size()) * sizeof(unsigned*)));
    P.d_targets = (unsigned**)p;
    CU(dev_alloc(h, &p, std::max<size_t>(1, P.recv_from.size()) * sizeof(int)));
    P.d_from = (int*)p;
    if (!targets.empty()) CU(cudaMemcpyAsync(P.d_targets, targets.data(), targets.size() * sizeof(unsigned*), cudaMemcpyHostToDevice, h->stream));
    if (!P.recv_from.empty()) CU(cudaMemcpyAsync(P.d_from, P.recv_from.data(), P.recv_from.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (h->opt.profile) {
        h->prof_ev.assign(4 * (size_t)h->m.T, nullptr);
        for (cudaEvent_t& e : h->prof_ev) CU(cudaEventCreate(&e));
    }
    P.attached = true;
    return SDPB_OK;
}

int sdpb_peer_traffic(const sdpb_handle* h, int64_t* bytes_out, int64_t* bytes_in) {
    if (!h || !h->peer.attached) return SDPB_ERR_STATE;
    if (bytes_out) *bytes_out = h->peer.bytes_out;
    if (bytes_in) *bytes_in = h->peer.bytes_in;
    return SDPB_OK;
}

int sdpb_period_profile(const sdpb_handle* h, double* ms) {
    if (!h || !ms) return SDPB_ERR_ARG;
    if (h->prof_ms.size() != 3 * (size_t)h->m.T) return SDPB_ERR_STATE;
    std::memcpy(ms, h->prof_ms.data(), h->prof_ms.size() * sizeof(double));
    return SDPB_OK;
}

// ---- one process, several GPUs ---------------------------------------------------------------------------------------
struct sdpb_group {
    std::vector<sdpb_handle*> shards;
    std::string err;
    double solve_ms = 0;
};

static thread_local std::string g_group_error;

const char* sdpb_group_last_error(const sdpb_group* g) { return g ? g->err.c_str() : g_group_error.c_str(); }

void sdpb_group_destroy(sdpb_group* g) {
    if (!g) return;
    for (sdpb_handle* h : g->shards)  // every stream drains before any table disappears
        if (h) { cudaSetDevice(h->device); cudaStreamSynchronize(h->stream); }
    for (sdpb_handle* h : g->shards) sdpb_destroy(h);
    delete g;
}

int sdpb_group_create(const sdpb_model* m, const sdpb_options* opt, const int* devices, int n, sdpb_group** out) {
    g_group_error.clear();
    if (!m || !devices || !out || n < 1 || n > kMaxPeers) { g_group_error = "bad argument"; return SDPB_ERR_ARG; }
    *out = nullptr;
    sdpb_group* g = new (std::nothrow) sdpb_group();
    if (!g) return SDPB_ERR_NOMEM;
    g->shards.assign(n, nullptr);
    auto fail = [&](int rc, const std::string& msg) { g_group_error = msg; sdpb_group_destroy(g); return rc; };
    for (int r = 0; r < n; r++) {
        sdpb_options o;
        std::memset(&o, 0, sizeof o);
        if (opt) o = *opt;
        o.struct_size = sizeof o;
        o.device = devices[r]; o.shard_rank = r; o.shard_count = n; o.stream = nullptr;
        const int rc = sdpb_create(m, &o, &g->shards[r]);
        if (rc != SDPB_OK) return fail(rc, "shard " + std::to_string(r) + ": " + sdpb_last_error(nullptr));
    }
    if (n > 1) {
        std::vector<unsigned char> blobs((size_t)n * SDPB_PEER_BLOB_BYTES);
        for (int r = 0; r < n; r++) {
            const int rc = sdpb_peer_export(g->shards[r], blobs.data() + (size_t)r * SDPB_PEER_BLOB_BYTES);
            if (rc != SDPB_OK) return fail(rc, "shard " + std::to_string(r) + ": " + g->shards[r]->err);
        }
        for (int r = 0; r < n; r++) {
            const int rc = sdpb_peer_attach(g->shards[r], blobs.data(), n);
            if (rc != SDPB_OK) return fail(rc, "shard " + std::to_string(r) + ": " + g->shards[r]->err);
        }
    }
    *out = g;
    return SDPB_OK;
}

sdpb_handle* sdpb_group_shard(sdpb_group* g, int rank) {
    return (g && rank >= 0 && rank < (int)g->shards.size()) ? g->shards[rank] : nullptr;
}

int sdpb_group_solve(sdpb_group* g) {
    if (!g) return SDPB_ERR_ARG;
    const int n = (int)g->shards.size();
    if (n == 1) {
        const int rc = sdpb_solve(g->shards[0]);
        if (rc != SDPB_OK) g->err = g->shards[0]->err;
        g->solve_ms = g->shards[0]->stats.solve_ms;
        return rc;
    }
    auto fail = [&](sdpb_handle* h, int rc) { g->err = "shard " + std::to_string(h->opt.shard_rank) + ": " + h->err; return rc; };
    const int T = g->shards[0]->m.T;
    for (sdpb_handle* h : g->shards) {
        if (cudaSetDevice(h->device) != cudaSuccess) { h->err = "cudaSetDevice failed"; return fail(h, SDPB_ERR_CUDA); }
        std::fill(h->solved.begin(), h->solved.end(), 0);
        h->stats = sdpb_stats{};
        cudaEventRecord(h->ev0, h->stream);
    }
    // one host thread feeds every shard's stream: for each period first every shard's kernels, pushes and flag, then
    // every shard's wait -- no wait is ever enqueued before the flag it waits for has been enqueued
    for (int t = T; t >= 1; t--) {
        for (sdpb_handle* h : g->shards) {
            cudaSetDevice(h->device);
            const int rc = enqueue_period_sharded(h, t, false);
            if (rc != SDPB_OK) return fail(h, rc);
        }
        if (t > 1)
            for (sdpb_handle* h : g->shards) {
                cudaSetDevice(h->device);
                const int rc = enqueue_period_exchange_wait(h);
                if (rc != SDPB_OK) return fail(h, rc);
                if (!h->prof_ev.empty()) cudaEventRecord(h->prof_ev[4 * (size_t)(t - 1) + 3], h->stream);
            }
    }
    g->solve_ms = 0;
    for (sdpb_handle* h : g->shards) {
        cudaSetDevice(h->device);
        cudaEventRecord(h->ev1, h->stream);
    }
    for (sdpb_handle* h : g->shards) {
        cudaSetDevice(h->device);
        if (cudaStreamSynchronize(h->stream) != cudaSuccess) { h->err = "stream synchronisation failed"; return fail(h, SDPB_ERR_CUDA); }
        float ms = 0;
        cudaEventElapsedTime(&ms, h->ev0, h->ev1);
        h->stats.solve_ms = h->stats.kernel_ms = ms;
        h->solve_count++;
        g->solve_ms = std::max(g->solve_ms, (double)ms);
        const int rc = finish_sharded(h);
        if (rc != SDPB_OK) return fail(h, rc);
    }
    return SDPB_OK;
}

int sdpb_group_value(sdpb_group* g, int period, const double* states, int n, double* v, double* q) {
    if (!g || !states || n < 0) return SDPB_ERR_ARG;
    sdpb_handle* h0 = g->shards[0];
    const int nd = h0->ndim;
    // route every state to the shard that owns it, one batched call per shard
    std::vector<std::vector<int>> who(g->shards.size());
    for (int i = 0; i < n; i++) {
        const long long idx = index_of_state(h0, states + (size_t)i * nd);
        if (idx < 0) { g->err = "state " + std::to_string(i) + " is not a grid point"; return SDPB_ERR_UNSOLVED; }
        size_t r = 0;
        while (r + 1 < g->shards.size() && idx >= g->shards[r]->hi) r++;
        who[r].push_back(i);
    }
    for (size_t r = 0; r < g->shards.size(); r++) {
        const std::vector<int>& ids = who[r];
        if (ids.empty()) continue;
        std::vector<double> st(ids.size() * nd), vv(ids.size()), qq(ids.size());
        for (size_t k = 0; k < ids.size(); k++) std::memcpy(&st[k * nd], states + (size_t)ids[k] * nd, nd * sizeof(double));
        const int rc = sdpb_value(g->shards[r], period, st.data(), (int)ids.size(), vv.data(), qq.data());
        if (rc != SDPB_OK) { g->err = g->shards[r]->err; return rc; }
        for (size_t k = 0; k < ids.size(); k++) { if (v) v[ids[k]] = vv[k]; if (q) q[ids[k]] = qq[k]; }
    }
    return SDPB_OK;
}

int sdpb_group_period_tables(sdpb_group* g, int period, double* V, double* Q) {
    if (!g) return SDPB_ERR_ARG;
    for (sdpb_handle* h : g->shards) {
        const int rc = sdpb_period_tables(h, period, V, Q);  // each shard fills its own block
        if (rc != SDPB_OK) { g->err = h->err; return rc; }
    }
    return SDPB_OK;
}

int sdpb_group_stats(const sdpb_group* g, sdpb_stats* s) {
    if (!g || !s) return SDPB_ERR_ARG;
    *s = sdpb_stats{};
    for (const sdpb_handle* h : g->shards) {
        s->evals += h->stats.evals; s->evals_executed += h->stats.evals_executed; s->fp64_ops += h->stats.fp64_ops;
        s->launches += h->stats.launches; s->kernel_used = h->stats.kernel_used;
        s->solve_ms = std::max(s->solve_ms, h->stats.solve_ms);
        s->kernel_ms = std::max(s->kernel_ms, h->stats.kernel_ms);
        s->exchange_ms = std::max(s->exchange_ms, h->stats.exchange_ms);
    }
    return SDPB_OK;
}

// ---- many small instances at once --------------------------------------------------------------------------------------
namespace {
struct BatchGraph {
    std::vector<sdpb_handle*> handles;
    cudaGraphExec_t exec = nullptr;
    cudaStream_t stream = nullptr;
    int device = 0;
    std::vector<sdpb_stats> stats;
};
std::mutex g_batch_mu;
std::vector<BatchGraph> g_batches;  // a handful per process: one per distinct handle list
}  // namespace

// sdpb_destroy: drop every remembered batch (and its graph) that contains the handle
static void forget_batches_of(sdpb_handle* h) {
    std::lock_guard<std::mutex> lk(g_batch_mu);
    for (size_t i = 0; i < g_batches.size();) {
        BatchGraph& b = g_batches[i];
        if (std::find(b.handles.begin(), b.handles.end(), h) != b.handles.end()) {
            if (b.exec) cudaGraphExecDestroy(b.exec);
            if (b.stream) { cudaStreamSynchronize(b.stream); cudaStreamDestroy(b.stream); }
            g_batches.erase(g_batches.begin() + (long)i);
        } else i++;
    }
}

int sdpb_solve_batch(sdpb_handle* const* handles, int n) {
    if (!handles || n < 1) return SDPB_ERR_ARG;
    sdpb_handle* h0 = handles[0];
    for (int i = 0; i < n; i++) {
        sdpb_handle* h = handles[i];
        if (!h) return SDPB_ERR_ARG;
        if (h->opt.shard_count != 1 || h->device != h0->device) { h->err = "sdpb_solve_batch needs unsharded handles of one device"; return SDPB_ERR_ARG; }
    }
    if (cudaSetDevice(h0->device) != cudaSuccess) return SDPB_ERR_CUDA;
    std::lock_guard<std::mutex> lk(g_batch_mu);
    BatchGraph* B = nullptr;
    for (BatchGraph& b : g_batches)
        if (b.handles.size() == (size_t)n && std::equal(b.handles.begin(), b.handles.end(), handles)) { B = &b; break; }
    if (B && B->exec) {  // replay: one launch for the whole batch
        for (int i = 0; i < n; i++) { handles[i]->stats = B->stats[i]; std::fill(handles[i]->solved.begin(), handles[i]->solved.end(), 1); }
        if (cudaGraphLaunch(B->exec, B->stream) != cudaSuccess || cudaStreamSynchronize(B->stream) != cudaSuccess) {
            h0->err = std::string("batch graph launch: ") + cudaGetErrorString(cudaGetLastError());
            return SDPB_ERR_CUDA;
        }
        return SDPB_OK;
    }
    if (!B) {
        // every instance gets 1/n of the GPU: no point in splitting its action range to fill all of it
        for (int i = 0; i < n; i++) handles[i]->tiled.batch = n;
        // first call with this list: plain solves (they create every scratch buffer); remember the list
        for (int i = 0; i < n; i++) { const int rc = sdpb_solve_async(handles[i]); if (rc != SDPB_OK) return rc; }
        for (int i = 0; i < n; i++) { const int rc = sdpb_sync(handles[i]); if (rc != SDPB_OK) return rc; }
        BatchGraph b;
        b.handles.assign(handles, handles + n);
        b.device = h0->device;
        g_batches.push_back(b);
        return SDPB_OK;
    }
    // second call: capture every handle's periods into one graph -- a fork from the batch stream into each handle's own
    // stream and a join back, so independent instances run side by side
    if (cudaStreamCreateWithFlags(&B->stream, cudaStreamNonBlocking) != cudaSuccess) return SDPB_ERR_CUDA;
    cudaGraph_t graph = nullptr;
    cudaEvent_t fork = nullptr;
    std::vector<cudaEvent_t> joins(n, nullptr);
    cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
    for (cudaEvent_t& e : joins) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    int rc = SDPB_OK;
    bool ok = cudaStreamBeginCapture(B->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
    if (ok) {
        ok = cudaEventRecord(fork, B->stream) == cudaSuccess;
        for (int i = 0; ok && i < n; i++) {
            sdpb_handle* h = handles[i];
            ok = cudaStreamWaitEvent(h->stream, fork, 0) == cudaSuccess;
            if (!ok) break;
            rc = enqueue_all_periods(h);
            if (rc != SDPB_OK) { ok = false; break; }
            ok = cudaEventRecord(joins[i], h->stream) == cudaSuccess && cudaStreamWaitEvent(B->stream, joins[i], 0) == cudaSuccess;
        }
        const cudaError_t e = cudaStreamEndCapture(B->stream, &graph);
        ok = ok && e == cudaSuccess && graph && cudaGraphInstantiate(&B->exec, graph, 0) == cudaSuccess;
        if (graph) cudaGraphDestroy(graph);
    }
    cudaEventDestroy(fork);
    for (cudaEvent_t e : joins) cudaEventDestroy(e);
    if (!ok) {
        cudaGetLastError();
        B->exec = nullptr;
        // capture is not possible here: plain solves again (and from now on)
        for (int i = 0; i < n; i++) { const int r2 = sdpb_solve_async(handles[i]); if (r2 != SDPB_OK) return r2; }
        for (int i = 0; i < n; i++) { const int r2 = sdpb_sync(handles[i]); if (r2 != SDPB_OK) return r2; }
        return SDPB_OK;
    }
    B->stats.resize(n);
    for (int i = 0; i < n; i++) B->stats[i] = handles[i]->stats;
    if (cudaGraphLaunch(B->exec, B->stream) != cudaSuccess || cudaStreamSynchronize(B->stream) != cudaSuccess) return SDPB_ERR_CUDA;
    return SDPB_OK;
}

int sdpb_trim_pool(int device) {
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) return SDPB_ERR_NO_DEVICE;
    if (device < 0 || device >= 64) return SDPB_ERR_ARG;
    std::lock_guard<std::mutex> lk(g_pool_mu);
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(device);
    for (const Slab& sl : g_slabs[device]) cudaFree(sl.p);
    g_slabs[device].clear();
    for (size_t i = 0; i < g_ipc_maps.size();) {
        if (g_ipc_maps[i].device == device) { cudaIpcCloseMemHandle(g_ipc_maps[i].p); g_ipc_maps.erase(g_ipc_maps.begin() + (long)i); }
        else i++;
    }
    cudaSetDevice(cur);
    cudaGetLastError();
    if (g_pools[device] && cudaMemPoolTrimTo(g_pools[device], 0) != cudaSuccess) { cudaGetLastError(); return SDPB_ERR_CUDA; }
    return SDPB_OK;
}

// ---- grid bounds for unclamped models (host arithmetic only) -----------------------------------------------------------
int sdpb_reachable_hull(const sdpb_model* m, const double* init_states, int n, double* inv_lo, double* inv_hi) {
    if (!m || !init_states || n < 1 || !inv_lo || !inv_hi || m->T < 1 || !m->pmf_len || !m->pmf_d) return SDPB_ERR_ARG;
    const bool cash = m->cost_kind != SDPB_COST_BACKORDER && m->cost_kind != SDPB_COST_STAFF;
    const bool two = m->cost_kind == SDPB_COST_CASH_TWO_PRODUCT;
    const int nd = 1 + (two ? 1 : 0) + (cash ? 1 : 0) + m->lead_time;
    // level before demand: x + (order, or the quantity already in the pipeline): in [x, x + max_order]
    const double amax = (double)m->max_order_idx * m->step;
    double lo = init_states[0], hi = init_states[0];
    for (int i = 0; i < n; i++) {
        const double* st = init_states + (size_t)i * nd;
        for (int k = 0; k < (two ? 2 : 1); k++) { lo = std::min(lo, st[k]); hi = std::max(hi, st[k]); }
    }
    double all_lo = lo, all_hi = hi;
    size_t off = 0;
    for (int t = 0; t < m->T; t++) {
        double dmin = m->pmf_d[off], dmax = m->pmf_d[off];
        for (int j = 0; j < m->pmf_len[t]; j++) { dmin = std::min(dmin, m->pmf_d[off + j]); dmax = std::max(dmax, m->pmf_d[off + j]); }
        if (two && m->pmf_d2)
            for (int j = 0; j < m->pmf_len[t]; j++) { dmin = std::min(dmin, m->pmf_d2[off + j]); dmax = std::max(dmax, m->pmf_d2[off + j]); }
        off += (size_t)m->pmf_len[t];
        if (t == m->T - 1 && !m->terminal_value) break;  // states of period T+1 exist only for the boundary function
        lo = lo - dmax;            // no order, largest demand
        hi = hi + amax - dmin;     // largest order (or pipeline quantity), smallest demand
        if (m->flags & SDPB_F_LOST_SALES) { lo = std::max(lo, 0.0); hi = std::max(hi, 0.0); }
        all_lo = std::min(all_lo, lo);
        all_hi = std::max(all_hi, hi);
    }
    *inv_lo = all_lo;
    *inv_hi = all_hi;
    return SDPB_OK;
}

int sdpb_stats_get(const sdpb_handle* h, sdpb_stats* s) {
    if (!h || !s) return SDPB_ERR_ARG;
    *s = h->stats;
    s->clipped_successors = h->reach_cnt[0];
    s->capped_action_sets = h->reach_cnt[1];
    s->cash_bound_hits = h->reach_cnt[2];
    return SDPB_OK;
}

}  // extern "C"
