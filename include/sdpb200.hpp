// sdpb200.hpp — C++17 host-side mirror of the reference's recursion classes over the C-ABI (sdpb200.h).
//
// The reference is Java (no JDK in the build image, INTEGRATION.md); this header is the compiled-language
// host side: the same class and member names, argument meaning and error behaviour as
//     sdp.inventory.State / Recursion            src/sdp/inventory/State.java, Recursion.java:33-186
//     sdp.inventory.LeadtimeState / LeadtimeRecursion   src/sdp/inventory/LeadtimeRecursion.java:28-75
//     sdp.cash.CashState / CashRecursion          src/sdp/cash/CashRecursion.java:39-220
//     sdp.cash.RiskRecursion                      src/sdp/cash/RiskRecursion.java:31-108
//     sdp.inventory.GetPmf (Poisson branch)       src/sdp/inventory/GetPmf.java:82-134
// with the three Java lambdas replaced by descriptor factories (one per reference driver, same parameter
// names as the driver's local variables).  Header-only; link with -lsdpb200.  tests/cpp_driver.cpp reads like
// CLSPTesting.main / CashConstraint.main / Leadtime.main and is checked against the oracle on a B200.
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "sdpb200.h"

namespace sdpb200 {

enum class OptDirection { MIN, MAX };  // sdp.inventory.GetPmf / Recursion.OptDirection

struct SdpbError : std::runtime_error {
    int code;
    SdpbError(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};

// double[][][] pmf of the reference: pmf[t][j] = {demand, probability}
using Pmf = std::vector<std::vector<std::array<double, 2>>>;

// ---- sdp.inventory.GetPmf, Poisson branch (GetPmf.java:88-119): support 0..(int) inverseF(q), probabilities
// prob(j) / (cdf(ub) - cdf(-1)).  SSJ's PoissonDist is replaced by lgamma-based sums, so the table agrees with
// SSJ to rounding, not bit for bit; solver parity is defined at the table boundary (DESIGN.md section 1).
class PoissonDist {
 public:
    explicit PoissonDist(double lambda) : lambda_(lambda) {}
    double prob(int k) const { return k < 0 ? 0.0 : std::exp(-lambda_ + k * std::log(lambda_) - std::lgamma(k + 1.0)); }
    double cdf(double x) const {
        double s = 0.0;
        for (int k = 0; k <= (int)std::floor(x); k++) s += prob(k);
        return s > 1.0 ? 1.0 : s;
    }
    double inverseF(double u) const {  // smallest k with cdf(k) >= u
        double s = 0.0;
        for (int k = 0;; k++) {
            s += prob(k);
            if (s >= u || k > 100000) return k;
        }
    }

 private:
    double lambda_;
};

class GetPmf {
 public:
    GetPmf(std::vector<PoissonDist> distributions, double truncationQuantile, double stepSize)
        : dists_(std::move(distributions)), q_(truncationQuantile), step_(stepSize) {}
    Pmf getpmf() const {
        Pmf pmf(dists_.size());
        for (size_t i = 0; i < dists_.size(); i++) {
            const double lb = 0.0, ub = (double)(int)dists_[i].inverseF(q_);
            const int n = (int)((ub - lb + 1) / step_);
            const double psum = dists_[i].cdf(ub) - dists_[i].cdf(lb - 1);
            for (int j = 0; j < n; j++) pmf[i].push_back({lb + j * step_, dists_[i].prob(j) / psum});
        }
        return pmf;
    }

 private:
    std::vector<PoissonDist> dists_;
    double q_, step_;
};

// ---- states (constructor argument order of the reference) ----
struct State {  // new State(period, iniInventory)
    int period;
    double iniInventory;
    int getPeriod() const { return period; }
    double getIniInventory() const { return iniInventory; }
};
struct LeadtimeState {  // new LeadtimeState(period, iniInventory, preQ)
    int period;
    double iniInventory, preQ;
};
struct CashState {  // new CashState(period, iniInventory, iniCash)
    int period;
    double iniInventory, iniCash;
    double getIniCash() const { return iniCash; }
};

// ---- descriptor + the arrays it points to ----
class Model {
 public:
    sdpb_model m;

    explicit Model(const Pmf& pmf) {
        std::memset(&m, 0, sizeof m);
        m.struct_size = (uint32_t)sizeof(sdpb_model);
        m.T = (int32_t)pmf.size();
        for (const auto& row : pmf) {
            len_.push_back((int32_t)row.size());
            for (const auto& dp : row) { d_.push_back(dp[0]); p_.push_back(dp[1]); }
        }
        m.gamma = 1.0; m.step = 1.0; m.quantiser = SDPB_Q_LONGDIV; m.q_mul = 1.0; m.q_div = 1.0;
        m.recursion = SDPB_REC_EXPECT; m.direction = SDPB_MIN; m.flags = SDPB_F_CLAMP_INV;
        fix();
    }
    Model(const Model& o) : m(o.m), len_(o.len_), d_(o.d_), p_(o.p_), price_t_(o.price_t_), vari_t_(o.vari_t_),
                            ovh_t_(o.ovh_t_), res_t_(o.res_t_), terminal_(o.terminal_) { fix(); }
    Model& operator=(const Model&) = delete;

    // FinalCash.BoundaryFuncton (FinalCash.java:16-18; consumed at CashRecursionV.java:125-128): the value of every grid
    // state of period T+1, in the library's state order (inventory outermost, cash innermost)
    Model& boundFinalCash(std::vector<double> table) { terminal_ = std::move(table); fix(); return *this; }

    // Leadtime.java:63-67 does not clamp: make the inventory axis the hull of what the recursion can reach
    Model& reachableHull(const std::vector<double>& initialState) {
        double lo = 0, hi = 0;
        if (sdpb_reachable_hull(&m, initialState.data(), 1, &lo, &hi) != SDPB_OK) throw SdpbError(SDPB_ERR_ARG, "sdpb_reachable_hull");
        m.inv_min = lo; m.inv_max = hi;
        return *this;
    }

    void setPerPeriod(const std::vector<double>* price, const std::vector<double>* vari, const std::vector<double>* ovh,
                      const std::vector<double>* reserve) {
        if (price) price_t_ = *price;
        if (vari) vari_t_ = *vari;
        if (ovh) ovh_t_ = *ovh;
        if (reserve) res_t_ = *reserve;
        fix();
    }

    // CLSPTesting.java:52-106 (also CLSP.java:251-272, LevelFitsS.java:74-102); G(y) pass: CLSPforDraw.java:147-170
    static Model inventory(OptDirection dir, const Pmf& pmf, double fixedOrderingCost, double variOrderingCost,
                           double holdingCost, double penaltyCost, double maxOrderQuantity, double minInventory,
                           double maxInventory, double stepSize = 1.0, bool isForDrawGy = false) {
        Model M(pmf);
        M.m.cost_kind = SDPB_COST_BACKORDER;
        M.m.direction = dir == OptDirection::MIN ? SDPB_MIN : SDPB_MAX;
        M.m.flags = SDPB_F_CLAMP_INV | (isForDrawGy ? SDPB_F_GY_MODE : 0);
        M.m.max_order_idx = (int32_t)(maxOrderQuantity / stepSize);
        M.m.inv_min = minInventory; M.m.inv_max = maxInventory; M.m.step = stepSize;
        M.m.fixed_cost = fixedOrderingCost; M.m.vari_cost = variOrderingCost;
        M.m.hold_cost = holdingCost; M.m.penalty_cost = penaltyCost;
        return M;
    }

    // Leadtime.java:33-81 (lead time 1, transition not clamped); leadTime 2 + clamp is config C4
    static Model leadtime(const Pmf& pmf, double fixedOrderingCost, double variOrderingCost, double holdingCost,
                          double penaltyCost, double maxOrderQuantity, double minInventory, double maxInventory,
                          double stepSize = 1.0, int leadTime = 1, bool clamp = false) {
        Model M = inventory(OptDirection::MIN, pmf, fixedOrderingCost, variOrderingCost, holdingCost, penaltyCost,
                            maxOrderQuantity, minInventory, maxInventory, stepSize);
        M.m.lead_time = leadTime;
        M.m.flags = clamp ? SDPB_F_CLAMP_INV : 0;
        return M;
    }

    // CashConstraint.java:44-133; quantiser round(w*10)/10.0 (:131) by default, (1, 1, long division) for
    // CashConstraintTesting.java:146
    static Model cashConstraint(const Pmf& pmf, double price, double variCost, double fixOrderCost, double holdingCost,
                                double salvageValue, double overheadCost, double overheadRate, double depositeRate,
                                double penaltyCost, double maxOrderQuantity, double minInventoryState,
                                double maxInventoryState, double minCashState, double maxCashState,
                                double discountFactor = 1.0, int quantiser = SDPB_Q_DIV, double qMul = 10.0,
                                double qDiv = 10.0) {
        Model M(pmf);
        M.m.cost_kind = SDPB_COST_CASH_DEPOSIT;
        M.m.direction = SDPB_MAX;
        M.m.flags = SDPB_F_CLAMP_INV | SDPB_F_LOST_SALES | SDPB_F_CASH_LIMITED_ACTIONS;
        M.m.max_order_idx = (int32_t)maxOrderQuantity;
        M.m.gamma = discountFactor;
        M.m.inv_min = minInventoryState; M.m.inv_max = maxInventoryState;
        M.m.cash_min = minCashState; M.m.cash_max = maxCashState;
        M.m.quantiser = quantiser; M.m.q_mul = qMul; M.m.q_div = qDiv;
        M.m.fixed_cost = fixOrderCost; M.m.vari_cost = variCost; M.m.hold_cost = holdingCost;
        M.m.penalty_cost = penaltyCost; M.m.price = price; M.m.salvage = salvageValue;
        M.m.deposit_rate = depositeRate; M.m.overhead_rate = overheadRate; M.m.overhead = overheadCost;
        M.m.reserve2 = fixOrderCost;
        const std::vector<double> res(pmf.size(), overheadCost);
        M.setPerPeriod(nullptr, nullptr, nullptr, &res);
        return M;
    }

    // cashSurvival.java:102-147: survival probability, per-period prices / costs, quantiser round(w*1)/1
    static Model cashSurvival(const Pmf& pmf, const std::vector<double>& price, const std::vector<double>& variCost,
                              const std::vector<double>& overheadCost, double salvageValue, double holdingCost,
                              double depositeRate, double fixOrderCost, double maxOrderQuantity, double minInventoryState,
                              double maxInventoryState, double minCashState, double maxCashState) {
        Model M = cashConstraint(pmf, 0.0, 0.0, fixOrderCost, holdingCost, salvageValue, 0.0, 0.0, depositeRate, 0.0,
                                 maxOrderQuantity, minInventoryState, maxInventoryState, minCashState, maxCashState, 1.0,
                                 SDPB_Q_LONGDIV, 1.0, 1.0);
        M.m.recursion = SDPB_REC_SURVIVAL;
        M.m.reserve2 = 0.0;
        M.res_t_.clear();
        M.setPerPeriod(&price, &variCost, &overheadCost, nullptr);
        return M;
    }

    // CashOverdraft.java:44-118: four-branch interest, quantiser round(w*10)/10 with LONG division (:116)
    static Model cashOverdraft(const Pmf& pmf, double price, double variCost, double fixOrderCost, double salvageValue,
                               const std::vector<double>& overheadCost, double r0, double r2, double r3, double limit,
                               double interestFreeAmount, double maxOrderQuantity, double minInventoryState,
                               double maxInventoryState, double minCashState, double maxCashState,
                               double discountFactor = 1.0) {
        Model M(pmf);
        M.m.cost_kind = SDPB_COST_CASH_OVERDRAFT;
        M.m.direction = SDPB_MAX;
        M.m.flags = SDPB_F_CLAMP_INV | SDPB_F_LOST_SALES;
        M.m.max_order_idx = (int32_t)maxOrderQuantity;
        M.m.gamma = discountFactor;
        M.m.inv_min = minInventoryState; M.m.inv_max = maxInventoryState;
        M.m.cash_min = minCashState; M.m.cash_max = maxCashState;
        M.m.quantiser = SDPB_Q_LONGDIV; M.m.q_mul = 10.0; M.m.q_div = 10.0;
        M.m.fixed_cost = fixOrderCost; M.m.vari_cost = variCost; M.m.price = price; M.m.salvage = salvageValue;
        M.m.r0 = r0; M.m.r2 = r2; M.m.r3 = r3; M.m.od_limit = limit; M.m.interest_free = interestFreeAmount;
        M.setPerPeriod(nullptr, nullptr, &overheadCost, nullptr);
        return M;
    }

 private:
    std::vector<int32_t> len_;
    std::vector<double> d_, p_, price_t_, vari_t_, ovh_t_, res_t_, terminal_;
    void fix() {
        m.terminal_value = terminal_.empty() ? nullptr : terminal_.data();
        m.pmf_len = len_.data(); m.pmf_d = d_.data(); m.pmf_p = p_.data();
        m.price_t = price_t_.empty() ? nullptr : price_t_.data();
        m.vari_cost_t = vari_t_.empty() ? nullptr : vari_t_.data();
        m.overhead_t = ovh_t_.empty() ? nullptr : ovh_t_.data();
        m.reserve_t = res_t_.empty() ? nullptr : res_t_.data();
    }
};

// ---- the engine every recursion class wraps: lazy whole-grid solve, then table look-ups ----
class Engine {
 public:
    explicit Engine(const Model& model, int device = -1, int kernel = SDPB_KERNEL_AUTO) : model_(model) {
        sdpb_options o;
        std::memset(&o, 0, sizeof o);
        o.struct_size = (uint32_t)sizeof o;
        o.device = device; o.shard_rank = 0; o.shard_count = 1; o.kernel = kernel;
        const int rc = sdpb_create(&model_.m, &o, &h_);
        if (rc != SDPB_OK) throw SdpbError(rc, std::string("sdpb_create: ") + sdpb_last_error(nullptr));
        sdpb_grid g;
        check(sdpb_grid_info(h_, &g));
        ndim_ = g.ndim;
    }
    // the same solve partitioned over several GPUs of this process (sdpb_group_*): bands of inventory rows, rows of
    // V_t handed from table to table through peer-mapped memory inside the library
    Engine(const Model& model, const std::vector<int>& devices, int kernel = SDPB_KERNEL_AUTO) : model_(model) {
        sdpb_options o;
        std::memset(&o, 0, sizeof o);
        o.struct_size = (uint32_t)sizeof o;
        o.kernel = kernel;
        const int rc = sdpb_group_create(&model_.m, &o, devices.data(), (int)devices.size(), &g_);
        if (rc != SDPB_OK) throw SdpbError(rc, std::string("sdpb_group_create: ") + sdpb_group_last_error(nullptr));
        sdpb_grid g;
        if (sdpb_grid_info(sdpb_group_shard(g_, 0), &g) != SDPB_OK) throw SdpbError(SDPB_ERR_ARG, "sdpb_grid_info");
        ndim_ = g.ndim;
    }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    ~Engine() { if (g_) sdpb_group_destroy(g_); else sdpb_destroy(h_); }

    // getExpectedValue / getAction of one state; the first call solves the whole horizon (Recursion.java:89-163
    // descends the whole reachable tree on its first call too)
    std::array<double, 2> valueAndAction(int period, const std::vector<double>& st) {
        if ((int)st.size() != ndim_) throw SdpbError(SDPB_ERR_ARG, "state has the wrong number of components");
        if (!solved_) {
            if (g_) { const int rc = sdpb_group_solve(g_); if (rc != SDPB_OK) throw SdpbError(rc, sdpb_group_last_error(g_)); }
            else check(sdpb_solve(h_));
            solved_ = true;
        }
        double v = 0.0, q = 0.0;
        if (g_) { const int rc = sdpb_group_value(g_, period, st.data(), 1, &v, &q); if (rc != SDPB_OK) throw SdpbError(rc, sdpb_group_last_error(g_)); }
        else check(sdpb_value(h_, period, st.data(), 1, &v, &q));
        if (period == 1) roots_.push_back(st);
        return {v, q};
    }
    bool solved() const { return solved_; }
    int ndim() const { return ndim_; }

    // getOptTable(): rows [period, state..., Q*] of the states the reference's memoisation would have visited
    // from the period-1 states queried so far, sorted by (period, state) (Recursion.java:169-186)
    std::vector<std::vector<double>> optTable() {
        if (!solved_ || roots_.empty()) throw SdpbError(SDPB_ERR_UNSOLVED, "getOptTable before getExpectedValue");
        if (g_) throw SdpbError(SDPB_ERR_STATE, "the visited-state table needs a single-GPU engine (sdpb_reach)");
        std::vector<double> flat;
        for (const auto& r : roots_) flat.insert(flat.end(), r.begin(), r.end());
        check(sdpb_reach(h_, flat.data(), (int)roots_.size()));
        size_t n = 0;
        check(sdpb_opt_table(h_, nullptr, &n));
        const size_t w = (size_t)ndim_ + 2;
        std::vector<double> buf(n * w);
        check(sdpb_opt_table(h_, buf.data(), &n));
        std::vector<std::vector<double>> rows(n, std::vector<double>(w));
        for (size_t i = 0; i < n; i++) std::copy(buf.begin() + i * w, buf.begin() + (i + 1) * w, rows[i].begin());
        return rows;
    }
    sdpb_stats stats() const { sdpb_stats s; sdpb_stats_get(h_, &s); return s; }
    sdpb_handle* handle() { return h_; }

    // Many independent single-GPU engines solved together (sdpb_solve_batch): the parameter sweeps of
    // CLSPTesting.java:57-61 build hundreds of small recursions one after the other; here their periods run side by
    // side as ONE CUDA graph (first call with a given list: plain solves; second: capture; later: replay).
    static void solveBatch(const std::vector<Engine*>& engines) {
        std::vector<sdpb_handle*> hs;
        for (Engine* e : engines) {
            if (e->g_) throw SdpbError(SDPB_ERR_ARG, "sdpb_solve_batch takes single-GPU engines");
            hs.push_back(e->h_);
        }
        if (hs.empty()) return;
        const int rc = sdpb_solve_batch(hs.data(), (int)hs.size());
        if (rc != SDPB_OK) throw SdpbError(rc, sdpb_last_error(hs[0]));
        for (Engine* e : engines) e->solved_ = true;
    }

 private:
    void check(int rc) const {
        if (rc != SDPB_OK) throw SdpbError(rc, sdpb_last_error(h_));
    }
    Model model_;
    sdpb_handle* h_ = nullptr;
    sdpb_group* g_ = nullptr;
    int ndim_ = 1;
    bool solved_ = false;
    std::vector<std::vector<double>> roots_;
};

// new Recursion(OptDirection, pmf, getFeasibleAction, stateTransition, immediateValue) -> new Recursion(model)
class Recursion {
 public:
    // `kernel`: SDPB_KERNEL_AUTO -- every kernel the library picks by itself is bit-identical to the Java loop -- or a
    // request, e.g. SDPB_KERNEL_COLLAPSED (G(y) per order-up-to level: ~1e-13 relative, opt-in)
    explicit Recursion(const Model& model, int device = -1, int kernel = SDPB_KERNEL_AUTO) : e_(model, device, kernel) {}
    Recursion(const Model& model, const std::vector<int>& devices) : e_(model, devices) {}
    double getExpectedValue(const State& s) { return e_.valueAndAction(s.period, {s.iniInventory})[0]; }
    // Recursion.java:165-167 unboxes a null for a state that was never solved; the mirror throws too
    double getAction(const State& s) {
        if (!e_.solved()) throw SdpbError(SDPB_ERR_UNSOLVED, "getAction on a state that was never solved");
        return e_.valueAndAction(s.period, {s.iniInventory})[1];
    }
    std::vector<std::vector<double>> getOptTable() { return e_.optTable(); }  // rows [t, x, Q*]
    void setTreeMapCacheAction() {}                                           // tables are always sorted
    Engine& engine() { return e_; }

 private:
    Engine e_;
};

class LeadtimeRecursion {  // LeadtimeRecursion.java:28-75
 public:
    explicit LeadtimeRecursion(const Model& model, int device = -1) : e_(model, device) {}
    LeadtimeRecursion(const Model& model, const std::vector<int>& devices) : e_(model, devices) {}
    std::vector<std::vector<double>> getOptTable() { return e_.optTable(); }  // rows [t, x, preQ, Q*]
    double getExpectedValue(const LeadtimeState& s) { return e_.valueAndAction(s.period, {s.iniInventory, s.preQ})[0]; }
    double getAction(const LeadtimeState& s) {
        if (!e_.solved()) throw SdpbError(SDPB_ERR_UNSOLVED, "getAction on a state that was never solved");
        return e_.valueAndAction(s.period, {s.iniInventory, s.preQ})[1];
    }
    Engine& engine() { return e_; }

 private:
    Engine e_;
};

class CashRecursion {  // CashRecursion.java:39-220
 public:
    explicit CashRecursion(const Model& model, int device = -1) : e_(model, device) {}
    CashRecursion(const Model& model, const std::vector<int>& devices) : e_(model, devices) {}
    double getExpectedValue(const CashState& s) { return e_.valueAndAction(s.period, {s.iniInventory, s.iniCash})[0]; }
    double getAction(const CashState& s) {
        if (!e_.solved()) throw SdpbError(SDPB_ERR_UNSOLVED, "getAction on a state that was never solved");
        return e_.valueAndAction(s.period, {s.iniInventory, s.iniCash})[1];
    }
    std::vector<std::vector<double>> getOptTable() { return e_.optTable(); }  // rows [t, x, w, Q*]
    Engine& engine() { return e_; }

 private:
    Engine e_;
};

class RiskRecursion {  // RiskRecursion.java:31-108: getSurvProb instead of getExpectedValue
 public:
    explicit RiskRecursion(const Model& model, int device = -1) : e_(model, device) {}
    double getSurvProb(const CashState& s) { return e_.valueAndAction(s.period, {s.iniInventory, s.iniCash})[0]; }
    double getAction(const CashState& s) {
        if (!e_.solved()) throw SdpbError(SDPB_ERR_UNSOLVED, "getAction on a state that was never solved");
        return e_.valueAndAction(s.period, {s.iniInventory, s.iniCash})[1];
    }
    Engine& engine() { return e_; }

 private:
    Engine e_;
};

// ---- no grid: the states the reference's recursion reaches from given period-1 states (sdpb_topdown_*) ----
// States, steps and demands need not be multiples of a power of two; an unclamped model needs no hull.
class TopDown {
 public:
    // `roots`: period-1 states in API order; scratchBytes = 0: the library's default expansion budget
    TopDown(const Model& model, const std::vector<std::vector<double>>& roots, int device = -1, uint32_t allow = 0,
            int64_t scratchBytes = 0) : model_(model) {
        sdpb_topdown_options o;
        std::memset(&o, 0, sizeof o);
        o.struct_size = (uint32_t)sizeof o;
        o.device = device; o.allow = allow; o.scratch_bytes = scratchBytes;
        std::vector<double> flat;
        for (const auto& r : roots) flat.insert(flat.end(), r.begin(), r.end());
        const int rc = sdpb_topdown_solve(&model_.m, &o, flat.data(), (int)roots.size(), &h_);
        if (rc != SDPB_OK) throw SdpbError(rc, std::string("sdpb_topdown_solve: ") + sdpb_topdown_last_error(nullptr));
    }
    TopDown(const TopDown&) = delete;
    TopDown& operator=(const TopDown&) = delete;
    ~TopDown() { sdpb_topdown_destroy(h_); }

    // (V, Q*) of a reached state; SdpbError(SDPB_ERR_UNSOLVED) for one that was not reached
    std::array<double, 2> valueAndAction(int period, const std::vector<double>& st) {
        if (st.size() != ndim_plus2() - 2) throw SdpbError(SDPB_ERR_ARG, "state has the wrong number of components");
        double v = 0.0, q = 0.0;
        check(sdpb_topdown_value(h_, period, st.data(), 1, &v, &q));
        return {v, q};
    }
    double value(int period, const std::vector<double>& st) { return valueAndAction(period, st)[0]; }
    // rows [period, state..., Q*] of every reached state in memo-map order (Recursion.java:169-186)
    std::vector<std::vector<double>> optTable() {
        size_t n = 0;
        check(sdpb_topdown_opt_table(h_, nullptr, &n));
        std::vector<double> buf(n * ndim_plus2());
        check(sdpb_topdown_opt_table(h_, buf.data(), &n));
        const size_t w = ndim_plus2();
        std::vector<std::vector<double>> rows(n, std::vector<double>(w));
        for (size_t i = 0; i < n; i++) std::copy(buf.begin() + i * w, buf.begin() + (i + 1) * w, rows[i].begin());
        return rows;
    }
    size_t nStates(int period) const {
        std::vector<int64_t> n((size_t)model_.m.T);
        check(sdpb_topdown_states(h_, n.data()));
        return (size_t)n.at((size_t)period - 1);
    }
    sdpb_stats stats() const { sdpb_stats s; check(sdpb_topdown_stats(h_, &s)); return s; }
    // getExpectedValue on API-order states of one period: solves only what no earlier call reached; a failure leaves
    // the handle as it was
    void extend(int period, const std::vector<std::vector<double>>& states) {
        std::vector<double> flat;
        for (const auto& r : states) {
            if (r.size() != ndim_plus2() - 2) throw SdpbError(SDPB_ERR_ARG, "state has the wrong number of components");
            flat.insert(flat.end(), r.begin(), r.end());
        }
        check(sdpb_topdown_extend(h_, period, flat.data(), (int)states.size()));
    }
    // Simulation.java:59-70 over demand sample paths (one row of T samples per path) -> per-path sums; every state a
    // path meets that was not reached is solved on the way and stays in the handle
    std::vector<double> simulate(const std::vector<double>& initState, const std::vector<std::vector<double>>& samples,
                                 double discount = 1.0) {
        if (initState.size() != ndim_plus2() - 2) throw SdpbError(SDPB_ERR_ARG, "state has the wrong number of components");
        std::vector<double> flat;
        for (const auto& r : samples) {
            if (r.size() != (size_t)model_.m.T) throw SdpbError(SDPB_ERR_ARG, "a sample path must have T demands");
            flat.insert(flat.end(), r.begin(), r.end());
        }
        std::vector<double> values(samples.size());
        check(sdpb_topdown_simulate(h_, initState.data(), flat.data(), (int)samples.size(), discount, values.data()));
        return values;
    }

 private:
    size_t ndim_plus2() const { return 3 + (model_.m.cost_kind != SDPB_COST_BACKORDER ? 1 : 0) + (size_t)model_.m.lead_time; }
    void check(int rc) const {
        if (rc != SDPB_OK) throw SdpbError(rc, sdpb_topdown_last_error(h_));
    }
    Model model_;
    sdpb_topdown* h_ = nullptr;
};

// ---- the two-product recursions (and CashConstraintTest's), over the states they reach (sdpb_reached_*) ----
// One memo for every call: every reached state can be queried, the handle extended with states of any period, and the
// policy rolled out.  States in API order: (x1, x2, preQ1, preQ2, cash) | (x1, x2, R) | (x1, x2, cash) | (x, cash).
class Reached {
 public:
    // `roots`: period-1 states (may be empty); the model's tables are copied.  scratchBytes > 0 replaces the free device
    // memory as the expansion budget
    Reached(const sdpb_reached_model& model, const std::vector<std::vector<double>>& roots, int device = -1,
            int64_t scratchBytes = 0) : T_(model.T), kind_(model.kind) {
        std::vector<double> flat = flatten(roots);
        const int rc = sdpb_reached_open(&model, device, scratchBytes, flat.data(), (int)roots.size(), &h_);
        if (rc != SDPB_OK) throw SdpbError(rc, std::string("sdpb_reached_open: ") + sdpb_reached_last_error());
    }
    Reached(const Reached&) = delete;
    Reached& operator=(const Reached&) = delete;
    ~Reached() { sdpb_reached_destroy(h_); }

    // (V, a1, a2) of a reached state; SdpbError(SDPB_ERR_UNSOLVED) for one that was not reached
    std::array<double, 3> valueAndAction(int period, const std::vector<double>& st) {
        if (st.size() != ndim()) throw SdpbError(SDPB_ERR_ARG, "state has the wrong number of components");
        std::array<double, 3> r{};
        check(sdpb_reached_value(h_, period, st.data(), 1, &r[0], &r[1], &r[2]));
        return r;
    }
    double value(int period, const std::vector<double>& st) { return valueAndAction(period, st)[0]; }
    // rows [period, state..., a1, a2] of every reached state in memo-map order
    std::vector<std::vector<double>> optTable() {
        size_t n = 0;
        check(sdpb_reached_opt_table(h_, nullptr, &n));
        const size_t w = ndim() + 3;
        std::vector<double> buf(n * w);
        check(sdpb_reached_opt_table(h_, buf.data(), &n));
        std::vector<std::vector<double>> rows(n, std::vector<double>(w));
        for (size_t i = 0; i < n; i++) std::copy(buf.begin() + i * w, buf.begin() + (i + 1) * w, rows[i].begin());
        return rows;
    }
    size_t nStates(int period) const {
        std::vector<int64_t> n((size_t)T_);
        check(sdpb_reached_states(h_, n.data()));
        return (size_t)n.at((size_t)period - 1);
    }
    sdpb_stats stats() const { sdpb_stats s; check(sdpb_reached_stats(h_, &s)); return s; }
    // getExpectedValue on API-order states of one period: solves only what no earlier call reached; a failure leaves
    // the handle as it was
    void extend(int period, const std::vector<std::vector<double>>& states) {
        std::vector<double> flat = flatten(states);
        check(sdpb_reached_extend(h_, period, flat.data(), (int)states.size()));
    }
    // the policy over demand sample paths (one row of T * nd samples per path, nd = 2 for two products, 1 for one) ->
    // per-path values; every state a path meets that was not reached is solved on the way and stays in the handle
    std::vector<double> simulate(const std::vector<double>& initState, const std::vector<std::vector<double>>& samples,
                                 double discount = 1.0) {
        if (initState.size() != ndim()) throw SdpbError(SDPB_ERR_ARG, "state has the wrong number of components");
        const size_t per = (size_t)T_ * (kind_ == SDPB_REACHED_CASH_ROUNDED ? 1 : 2);
        std::vector<double> flat;
        for (const auto& r : samples) {
            if (r.size() != per) throw SdpbError(SDPB_ERR_ARG, "a sample path must have T * nd demands");
            flat.insert(flat.end(), r.begin(), r.end());
        }
        std::vector<double> values(samples.size());
        check(sdpb_reached_simulate(h_, initState.data(), flat.data(), (int)samples.size(), discount, values.data()));
        return values;
    }

 private:
    size_t ndim() const { return kind_ == SDPB_REACHED_MULTILEAD ? 5 : kind_ == SDPB_REACHED_CASH_ROUNDED ? 2 : 3; }
    std::vector<double> flatten(const std::vector<std::vector<double>>& states) const {
        std::vector<double> flat;
        for (const auto& r : states) {
            if (r.size() != ndim()) throw SdpbError(SDPB_ERR_ARG, "state has the wrong number of components");
            flat.insert(flat.end(), r.begin(), r.end());
        }
        return flat;
    }
    void check(int rc) const {
        if (rc != SDPB_OK) throw SdpbError(rc, sdpb_reached_last_error());
    }
    int T_, kind_;
    sdpb_reached* h_ = nullptr;
};

// Recursion / LeadtimeRecursion / CashRecursion / RiskRecursion access over TopDown, with states given as API-order
// vectors: getExpectedValue on a new period-1 state extends the solve with that root (the memo maps grow the same way;
// states a roll-out over engine() added stay); getAction / getExpectedValue of a later-period state that was not
// reached throws SDPB_ERR_UNSOLVED.
class TopDownRecursion {
 public:
    explicit TopDownRecursion(const Model& model, int device = -1, uint32_t allow = 0)
        : model_(model), device_(device), allow_(allow) {}
    double getExpectedValue(int period, const std::vector<double>& st) {
        if (period == 1 && std::find(roots_.begin(), roots_.end(), st) == roots_.end()) {
            // if this throws, the roots and the solve stay as they were
            if (td_) td_->extend(1, {st});
            else td_.reset(new TopDown(model_, {st}, device_, allow_));
            roots_.push_back(st);
        }
        return engine().value(period, st);
    }
    double getAction(int period, const std::vector<double>& st) { return engine().valueAndAction(period, st)[1]; }
    double getExpectedValue(const State& s) { return getExpectedValue(s.period, {s.iniInventory}); }
    double getAction(const State& s) { return getAction(s.period, {s.iniInventory}); }
    double getExpectedValue(const LeadtimeState& s) { return getExpectedValue(s.period, {s.iniInventory, s.preQ}); }
    double getAction(const LeadtimeState& s) { return getAction(s.period, {s.iniInventory, s.preQ}); }
    double getExpectedValue(const CashState& s) { return getExpectedValue(s.period, {s.iniInventory, s.iniCash}); }
    double getSurvProb(const CashState& s) { return getExpectedValue(s); }
    double getAction(const CashState& s) { return getAction(s.period, {s.iniInventory, s.iniCash}); }
    std::vector<std::vector<double>> getOptTable() { return engine().optTable(); }
    TopDown& engine() {
        if (!td_) throw SdpbError(SDPB_ERR_UNSOLVED, "no period-1 state has been solved");
        return *td_;
    }

 private:
    Model model_;
    int device_;
    uint32_t allow_;
    std::vector<std::vector<double>> roots_;
    std::unique_ptr<TopDown> td_;
};

}  // namespace sdpb200
