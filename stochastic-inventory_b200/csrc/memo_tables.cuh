// memo_tables.cuh — the memo tables of a handle that solves a model over the states it reaches, shared by the top-down
// engine (topdown.cu) and the reached-state engine (reached.cu).
//
// Per period t the tables hold the reached states F_t, sorted by key, with their value V_t and action index Q_t.  An
// extension builds the new states N_t of the periods it touches into a stage (the engine's forward pass), solves them
// against the merged tables of the next period (the engine's backward kernels), merges (N_t, V, Q) into (F_t, V_t, Q_t)
// by key, and commits the merged tables only at the end, so that a failed extension leaves the handle as it was.  The
// queries and the policy roll-out search the same tables.
//
// An engine brings its key through a traits class K:
//   K::Key                    the key type, trivially copyable
//   K::Less, K::Eq            host / device comparators; the tables are sorted by Less
//   K::lower(F, n, k)         (device) the first index of F[0, n) whose key is not less than k
// and, to the roll-out, a step (see memo_simulate).  Every shared function returns an sdpb_status and, on failure,
// leaves its message in `err`, the engine's last-error string.
#pragma once

#include <cuda_runtime.h>
#include <thrust/execution_policy.h>
#include <thrust/iterator/zip_iterator.h>
#include <thrust/merge.h>
#include <thrust/tuple.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <exception>
#include <string>
#include <vector>

#include "../../include/sdpb200.h"

namespace memo {

inline int fail(std::string& err, int rc, const std::string& msg) {
    err = msg;
    return rc;
}

struct DevBuf {  // a scratch allocation released when it goes out of scope
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    bool alloc(size_t bytes) {
        if (p) { cudaFree(p); p = nullptr; }
        if (cudaMalloc(&p, bytes > 0 ? bytes : 16) != cudaSuccess) { cudaGetLastError(); p = nullptr; return false; }
        return true;
    }
};

// a right-sized table of n entries (at least one, so that an empty table is not a null pointer)
template <class P>
bool alloc(P*& p, long long n) {
    if (cudaMalloc((void**)&p, (size_t)std::max(n, 1ll) * sizeof(P)) == cudaSuccess) return true;
    cudaGetLastError();
    p = nullptr;
    return false;
}

// sorted by K::Less, each key once: the canonical form of a set of roots
template <class K>
void canonical(std::vector<typename K::Key>& v) {
    std::sort(v.begin(), v.end(), typename K::Less());
    v.erase(std::unique(v.begin(), v.end(), typename K::Eq()), v.end());
}

// The tables of one handle, its stream, the events that time an extension or a roll-out, and its statistics.
template <class K>
struct Tables {
    typedef typename K::Key Key;
    std::vector<Key*> F;      // [T] reached states, sorted
    std::vector<double*> V;   // [T]
    std::vector<int*> Q;      // [T] action index
    std::vector<long long> nF;
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
    sdpb_stats stats{};

    Tables() = default;
    Tables(const Tables&) = delete;
    Tables& operator=(const Tables&) = delete;
    // on the handle's device
    ~Tables() {
        for (Key* p : F) cudaFree(p);
        for (double* p : V) cudaFree(p);
        for (int* p : Q) cudaFree(p);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (e2) cudaEventDestroy(e2);
        if (stream) cudaStreamDestroy(stream);
        cudaGetLastError();
    }
    // T empty periods, the stream and the events, on the current device
    int open(int T, std::string& err) {
        F.assign(T, nullptr);
        V.assign(T, nullptr);
        Q.assign(T, nullptr);
        nF.assign(T, 0);
        if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&e0) != cudaSuccess ||
            cudaEventCreate(&e1) != cudaSuccess || cudaEventCreate(&e2) != cudaSuccess)
            return fail(err, SDPB_ERR_CUDA, "stream / event creation failed");
        return SDPB_OK;
    }
};

// What one extension builds, owned here until it is committed to the handle: per period the new states N_t with their
// V / Q, and the merged tables F_t u N_t.  Whatever is still owned when the stage goes out of scope is freed, so an
// extension that fails leaves the handle as it found it.
template <class K>
struct Stage {
    typedef typename K::Key Key;
    std::vector<Key*> N, MF;
    std::vector<double*> VN, MV;
    std::vector<int*> QN, MQ;
    std::vector<long long> nN, nM;
    explicit Stage(int T)
        : N(T, nullptr), MF(T, nullptr), VN(T, nullptr), MV(T, nullptr), QN(T, nullptr), MQ(T, nullptr), nN(T, 0), nM(T, 0) {}
    ~Stage() {
        for (size_t k = 0; k < N.size(); k++) {
            cudaFree(N[k]); cudaFree(MF[k]); cudaFree(VN[k]); cudaFree(MV[k]); cudaFree(QN[k]); cudaFree(MQ[k]);
        }
    }
};

// The second half of an extension from period p, after the engine's forward pass filled sg.N / sg.nN and counted
// `evals` evaluations and `capped` capped action sets (e0 was recorded before the forward pass).  For t = T .. p:
// backward(t, N, n, Fn, Vn, nFn, V, Q) launches the engine's backward kernel(s) for the n new states N of period t
// against the sorted (Fn, Vn) of period t + 1 (nFn states; none when t == T) into (V, Q) and returns how many launches it
// made, or a status < 0 with its message stored; then the new states are merged into the period's tables by key.  The
// merged tables replace the handle's once all of them are built.
template <class K, class Backward>
int commit(Tables<K>& mt, Stage<K>& sg, int p, double evals, double capped, Backward backward, std::string& err) {
    const int T = (int)mt.F.size();
    cudaStream_t st = mt.stream;
    if (cudaEventRecord(mt.e1, st) != cudaSuccess) return fail(err, SDPB_ERR_CUDA, "cudaEventRecord failed");
    int launches = 0;
    for (int t = T; t >= p; t--) {
        const int k = t - 1;
        const long long n = sg.nN[k], no = mt.nF[k];
        if (n == 0) continue;
        if (!alloc(sg.VN[k], n) || !alloc(sg.QN[k], n)) return fail(err, SDPB_ERR_NOMEM, "allocation of the value tables failed");
        const bool nxt = t < T, nxt_new = nxt && sg.nN[k + 1] > 0;
        const int l = backward(t, (const typename K::Key*)sg.N[k], n, nxt ? (nxt_new ? sg.MF[k + 1] : mt.F[k + 1]) : nullptr,
                               nxt ? (nxt_new ? sg.MV[k + 1] : mt.V[k + 1]) : nullptr,
                               nxt ? (nxt_new ? sg.nM[k + 1] : mt.nF[k + 1]) : 0, sg.VN[k], sg.QN[k]);
        if (l < 0) return l;
        launches += l;
        if (cudaGetLastError() != cudaSuccess) return fail(err, SDPB_ERR_CUDA, "backward launch failed");
        sg.nM[k] = no + n;
        if (no == 0) {  // nothing to merge with: the new tables are the merged ones
            std::swap(sg.MF[k], sg.N[k]);
            std::swap(sg.MV[k], sg.VN[k]);
            std::swap(sg.MQ[k], sg.QN[k]);
            continue;
        }
        if (!alloc(sg.MF[k], no + n) || !alloc(sg.MV[k], no + n) || !alloc(sg.MQ[k], no + n))
            return fail(err, SDPB_ERR_NOMEM, "allocation of the merged tables of period " + std::to_string(t) + " failed");
        try {  // the two key sets are disjoint: a merge by key keeps every row
            thrust::merge_by_key(thrust::cuda::par.on(st), mt.F[k], mt.F[k] + no, sg.N[k], sg.N[k] + n,
                                 thrust::make_zip_iterator(thrust::make_tuple(mt.V[k], mt.Q[k])),
                                 thrust::make_zip_iterator(thrust::make_tuple(sg.VN[k], sg.QN[k])), sg.MF[k],
                                 thrust::make_zip_iterator(thrust::make_tuple(sg.MV[k], sg.MQ[k])), typename K::Less());
        } catch (const std::exception& ex) {
            return fail(err, SDPB_ERR_CUDA, std::string("merge: ") + ex.what());
        }
    }
    if (cudaEventRecord(mt.e2, st) != cudaSuccess || cudaEventSynchronize(mt.e2) != cudaSuccess)
        return fail(err, SDPB_ERR_CUDA, std::string("backward pass: ") + cudaGetErrorString(cudaGetLastError()));
    for (int k = p - 1; k < T; k++) {  // commit; the stage frees the tables it replaces
        if (sg.nN[k] == 0) continue;
        std::swap(mt.F[k], sg.MF[k]);
        std::swap(mt.V[k], sg.MV[k]);
        std::swap(mt.Q[k], sg.MQ[k]);
        mt.nF[k] = sg.nM[k];
    }
    float solve = 0, kern = 0;
    cudaEventElapsedTime(&solve, mt.e0, mt.e2);
    cudaEventElapsedTime(&kern, mt.e1, mt.e2);
    mt.stats.evals += evals;
    mt.stats.evals_executed += evals;
    mt.stats.capped_action_sets += capped;
    mt.stats.solve_ms = solve;
    mt.stats.kernel_ms = kern;
    mt.stats.launches = launches;
    return SDPB_OK;
}

// batched lookup: (V, action index) of each query key, action index -2 when the state is not in the sorted table F
template <class K>
__global__ void memo_query(const typename K::Key* __restrict__ F, const long long n, const double* __restrict__ V,
                           const int* __restrict__ Q, const typename K::Key* __restrict__ q, const int nq,
                           double* __restrict__ v, int* __restrict__ qi) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const typename K::Key k = q[i];
    const long long at = K::lower(F, n, k);
    const bool hit = at < n && typename K::Eq()(F[at], k);
    v[i] = hit ? V[at] : 0.0;
    qi[i] = hit ? Q[at] : -2;
}

// (V, action index) of the keys of period `period`; SDPB_ERR_UNSOLVED when one of them was not reached
template <class K>
int lookup(const Tables<K>& mt, int period, const std::vector<typename K::Key>& keys, std::vector<double>& v,
           std::vector<int>& qi, std::string& err) {
    typedef typename K::Key Key;
    const int n = (int)keys.size();
    DevBuf kq, vq, aq;
    if (!kq.alloc(keys.size() * sizeof(Key)) || !vq.alloc((size_t)n * sizeof(double)) || !aq.alloc((size_t)n * sizeof(int)))
        return fail(err, SDPB_ERR_NOMEM, "allocation failed");
    v.resize((size_t)n);
    qi.resize((size_t)n);
    cudaStream_t st = mt.stream;
    if (cudaMemcpyAsync(kq.p, keys.data(), keys.size() * sizeof(Key), cudaMemcpyHostToDevice, st) != cudaSuccess)
        return fail(err, SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
    memo_query<K><<<(n + 127) / 128, 128, 0, st>>>(mt.F[period - 1], mt.nF[period - 1], mt.V[period - 1], mt.Q[period - 1],
                                                  (const Key*)kq.p, n, (double*)vq.p, (int*)aq.p);
    if (cudaGetLastError() != cudaSuccess ||
        cudaMemcpyAsync(v.data(), vq.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaMemcpyAsync(qi.data(), aq.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
        return fail(err, SDPB_ERR_CUDA, std::string("query: ") + cudaGetErrorString(cudaGetLastError()));
    for (int i = 0; i < n; i++)
        if (qi[i] == -2)
            return fail(err, SDPB_ERR_UNSOLVED, "state " + std::to_string(i) + " was not reached in period " + std::to_string(period));
    return SDPB_OK;
}

// The getOptTable() rows of every reached state, period by period in key order, w doubles each: row(t, key, v, qi, out)
// writes the row of one state.  *nrows: the rows `rows` holds; without `rows`, the number of reached states.
template <class K, class Row>
int opt_table(const Tables<K>& mt, double* rows, size_t* nrows, int w, Row row, std::string& err) {
    size_t total = 0;
    for (long long n : mt.nF) total += (size_t)n;
    if (!rows) { *nrows = total; return SDPB_OK; }
    if (*nrows < total) return fail(err, SDPB_ERR_ARG, "rows holds fewer than the reached states");
    std::vector<typename K::Key> k;
    std::vector<double> v;
    std::vector<int> qi;
    size_t r = 0;
    for (int t = 1; t <= (int)mt.nF.size(); t++) {
        const size_t n = (size_t)mt.nF[t - 1];
        k.resize(n);
        v.resize(n);
        qi.resize(n);
        if (cudaMemcpyAsync(k.data(), mt.F[t - 1], n * sizeof(typename K::Key), cudaMemcpyDeviceToHost, mt.stream) != cudaSuccess ||
            cudaMemcpyAsync(v.data(), mt.V[t - 1], n * sizeof(double), cudaMemcpyDeviceToHost, mt.stream) != cudaSuccess ||
            cudaMemcpyAsync(qi.data(), mt.Q[t - 1], n * sizeof(int), cudaMemcpyDeviceToHost, mt.stream) != cudaSuccess ||
            cudaStreamSynchronize(mt.stream) != cudaSuccess)
            return fail(err, SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
        for (size_t i = 0; i < n; i++, r++) row(t, k[i], v[i], qi[i], rows + r * w);
    }
    *nrows = total;
    return SDPB_OK;
}

// One thread per path of act[0, na): from where the path stands (period per[i], state key[i], partial sum sum[i]) --
// the state's action and value, the samples of period t (nd per period), the step, sum += discount^(t-1) c -- until it
// ends (values[i] = sum) or meets a state the handle has not reached.  There it writes (path, t, state) to the next slot
// of the stall list, keeps its period, state and partial sum, and stops; the host extends the handle with the stalled
// states and relaunches the stalled paths.
//
// step(t, s, qi, v, smp, c) sets c to the cost of period t for a path at state s, whose action index is qi and value v,
// under the samples smp of the period, and s to the successor state when t < T.  It returns true when c is the path's
// whole value instead of a cost to add (the V / Pi form at t == T).
template <class K, class Step>
__global__ void __launch_bounds__(128) memo_simulate(const __grid_constant__ Step step, const int T,
                                                     const typename K::Key* const* __restrict__ tF,
                                                     const double* const* __restrict__ tV, const int* const* __restrict__ tQ,
                                                     const long long* __restrict__ tn, const double* __restrict__ samples,
                                                     const int nd, const double* __restrict__ pw, const int* __restrict__ act,
                                                     const int na, typename K::Key* __restrict__ key, int* __restrict__ per,
                                                     double* __restrict__ sum, double* __restrict__ values,
                                                     int* __restrict__ stall_n, int* __restrict__ stall_path,
                                                     int* __restrict__ stall_t, typename K::Key* __restrict__ stall_key) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= na) return;
    const int i = act[k];
    typename K::Key s = key[i];
    double acc = sum[i];
    for (int t = per[i]; t <= T; t++) {
        const typename K::Key* __restrict__ F = tF[t - 1];
        const long long n = tn[t - 1];
        const long long at = K::lower(F, n, s);
        if (at >= n || !typename K::Eq()(F[at], s)) {
            key[i] = s;
            per[i] = t;
            sum[i] = acc;
            const int slot = atomicAdd(stall_n, 1);
            stall_path[slot] = i;
            stall_t[slot] = t;
            stall_key[slot] = s;
            return;
        }
        double c;
        if (step(t, s, tQ[t - 1][at], tV[t - 1][at], samples + ((size_t)i * T + (t - 1)) * nd, c)) acc = c;
        else acc += pw[t - 1] * c;
    }
    values[i] = acc;
}

// The policy roll-out of n paths from the state k0 of period 1 over the handle, with the engine's step: samples holds nd
// demands per path and period.  extend(p, roots) is the engine's extension from period p (roots[t - 1]: the canonical
// roots of period t), which stores its own message.  The first extension is getExpectedValue(k0), as the reference's
// Simulation asks for it first; then every round extends the handle with the states the stalled paths stand on and
// relaunches those paths.
template <class K, class Step, class Extend>
int rollout(Tables<K>& mt, const Step& step, const typename K::Key& k0, const double* samples, int n, int nd,
            double discount, Extend extend, double* values, std::string& err) {
    typedef typename K::Key Key;
    const int T = (int)mt.F.size();
    const auto w0 = std::chrono::steady_clock::now();
    std::vector<std::vector<Key>> roots((size_t)T);
    roots[0].push_back(k0);
    int rc = extend(1, roots);
    if (rc != SDPB_OK) return rc;

    cudaStream_t st = mt.stream;
    const size_t N = (size_t)n;
    std::vector<double> pw((size_t)T);
    for (int t = 0; t < T; t++) pw[t] = std::pow(discount, (double)t);  // Math.pow(discountFactor, t)
    std::vector<Key> key0(N, k0);
    std::vector<int> per0(N, 1), act0(N);
    for (int i = 0; i < n; i++) act0[i] = i;
    DevBuf smp_b, pw_b, key_b, per_b, sum_b, val_b, act_b[2], st_b, sk_b, sn_b, tab_b;
    if (!smp_b.alloc(N * T * nd * sizeof(double)) || !pw_b.alloc(T * sizeof(double)) || !key_b.alloc(N * sizeof(Key)) ||
        !per_b.alloc(N * sizeof(int)) || !sum_b.alloc(N * sizeof(double)) || !val_b.alloc(N * sizeof(double)) ||
        !act_b[0].alloc(N * sizeof(int)) || !act_b[1].alloc(N * sizeof(int)) || !st_b.alloc(N * sizeof(int)) ||
        !sk_b.alloc(N * sizeof(Key)) || !sn_b.alloc(sizeof(int)) || !tab_b.alloc((size_t)T * 4 * 8))
        return fail(err, SDPB_ERR_NOMEM, "allocation of the roll-out buffers failed");
    const Key** dF = (const Key**)tab_b.p;
    const double** dV = (const double**)(dF + T);
    const int** dQ = (const int**)(dV + T);
    long long* dn = (long long*)(dQ + T);
    if (cudaMemcpyAsync(smp_b.p, samples, N * T * nd * sizeof(double), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(pw_b.p, pw.data(), T * sizeof(double), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(key_b.p, key0.data(), N * sizeof(Key), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(per_b.p, per0.data(), N * sizeof(int), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(act_b[0].p, act0.data(), N * sizeof(int), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemsetAsync(sum_b.p, 0, N * sizeof(double), st) != cudaSuccess)
        return fail(err, SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
    std::vector<const void*> tab((size_t)T * 4);
    std::vector<int> stall_t;
    std::vector<Key> stall_k;
    float kern = 0;
    int rounds = 0, na = n, cur = 0;
    while (na > 0) {
        // the tables move when an extension merges new states in: hand the kernel the current ones
        for (int t = 0; t < T; t++) {
            tab[t] = mt.F[t];
            tab[T + t] = mt.V[t];
            tab[2 * T + t] = mt.Q[t];
            std::memcpy(&tab[3 * T + t], &mt.nF[t], sizeof(long long));
        }
        int ns = 0;
        if (cudaMemcpyAsync(tab_b.p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, st) != cudaSuccess ||
            cudaMemsetAsync(sn_b.p, 0, sizeof(int), st) != cudaSuccess || cudaEventRecord(mt.e1, st) != cudaSuccess)
            return fail(err, SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
        memo_simulate<K, Step><<<(na + 127) / 128, 128, 0, st>>>(step, T, dF, dV, dQ, dn, (const double*)smp_b.p, nd,
                                                                 (const double*)pw_b.p, (const int*)act_b[cur].p, na,
                                                                 (Key*)key_b.p, (int*)per_b.p, (double*)sum_b.p,
                                                                 (double*)val_b.p, (int*)sn_b.p, (int*)act_b[1 - cur].p,
                                                                 (int*)st_b.p, (Key*)sk_b.p);
        if (cudaGetLastError() != cudaSuccess) return fail(err, SDPB_ERR_CUDA, "roll-out launch failed");
        if (cudaEventRecord(mt.e2, st) != cudaSuccess ||
            cudaMemcpyAsync(&ns, sn_b.p, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            return fail(err, SDPB_ERR_CUDA, std::string("roll-out: ") + cudaGetErrorString(cudaGetLastError()));
        float ms = 0;
        cudaEventElapsedTime(&ms, mt.e1, mt.e2);
        kern += ms;
        rounds++;
        if (ns == 0) break;
        // the states the stalled paths stand on become the roots of one extension (getExpectedValue(state))
        stall_t.resize((size_t)ns);
        stall_k.resize((size_t)ns);
        if (cudaMemcpyAsync(stall_t.data(), st_b.p, (size_t)ns * sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaMemcpyAsync(stall_k.data(), sk_b.p, (size_t)ns * sizeof(Key), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            return fail(err, SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
        std::vector<std::vector<Key>> r((size_t)T);
        int p = T;
        for (int j = 0; j < ns; j++) {
            r[stall_t[j] - 1].push_back(stall_k[j]);
            p = std::min(p, stall_t[j]);
        }
        for (auto& v : r) canonical<K>(v);
        rc = extend(p, r);
        if (rc != SDPB_OK) return rc;
        na = ns;
        cur = 1 - cur;
    }
    if (cudaMemcpyAsync(values, val_b.p, N * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
        return fail(err, SDPB_ERR_CUDA, "cudaMemcpyAsync failed");
    mt.stats.solve_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - w0).count();
    mt.stats.kernel_ms = kern;
    mt.stats.launches = rounds;
    return SDPB_OK;
}

}  // namespace memo
