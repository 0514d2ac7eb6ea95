// CPU references for the reached-state handle (sdpb_reached_open / _extend / _value / _opt_table / _simulate); test
// infrastructure, never linked into libsdpb200.so.  This file includes oracle/sdp_oracle.cpp unchanged and drives its
// memoised recursions in a new order: kind 0 on the file's TopDown with the MultiLead lambdas (as oracle_multi_lead
// does), kinds 1-3 on its ReachedTopDown.  Both take the sdpb_reached_model the library takes.
// Built by tests/reached_oracle.py with the oracle's flags (-ffp-contract=off: Java never fuses multiply-add).
#include "../oracle/sdp_oracle.cpp"

#include <memory>
#include <stdexcept>

namespace {

// One memo of the reference's recursion for `m`, whatever its kind.  States and rows in API order.
struct Memo {
    const sdpb_reached_model& m;
    std::vector<int> lens;
    // kind 0
    MultiLead ml;
    std::vector<int32_t> len0;
    std::vector<double> pd, pp;
    sdpb_model dm;
    Model M;
    std::unique_ptr<TopDown> td;
    // kinds 1-3
    RParamsO P;
    std::unique_ptr<ReachedTopDown> rt;

    explicit Memo(const sdpb_reached_model& mm) : m(mm) {
        const int T = m.T, nD = m.n_demands;
        for (int t = 0; t < T; t++) lens.push_back(m.n_demands_t ? m.n_demands_t[t] : nD);
        if (m.kind == SDPB_REACHED_MULTILEAD) {
            ml.Qbound = m.q_bound;
            for (int k = 0; k < 2; k++) { ml.price[k] = m.price[k]; ml.variCost[k] = m.vari_cost[k]; ml.salValueUnit[k] = m.salvage[k]; }
            ml.r0 = m.r0; ml.r1 = m.r1; ml.r2 = m.r2; ml.limit = m.limit; ml.interestFreeAmount = m.interest_free;
            ml.minInventoryState = m.min_inv; ml.maxInventoryState = m.max_inv;
            ml.minCashState = m.min_cash; ml.maxCashState = m.max_cash;
            ml.overheadCost.assign(m.overhead_t, m.overhead_t + T);
            // the loop hands the lambdas the flat index j of a demand pair; MultiLead keeps one pair table for every
            // period, so the periods must share it (the callers' pmfs do)
            for (int j = 0; j < lens[0]; j++) { ml.d1.push_back((int)m.d1[j]); ml.d2.push_back((int)m.d2[j]); }
            for (int t = 0; t < T; t++) {
                if (lens[t] != lens[0]) throw std::runtime_error("kind 0: every period must have the same demand pairs");
                for (int j = 0; j < lens[t]; j++) {
                    if (m.d1[t * nD + j] != m.d1[j] || m.d2[t * nD + j] != m.d2[j])
                        throw std::runtime_error("kind 0: every period must have the same demand pairs");
                    pd.push_back((double)j);
                    pp.push_back(m.p[t * nD + j]);
                }
                len0.push_back(lens[t]);
            }
            std::memset(&dm, 0, sizeof dm);
            dm.T = T; dm.direction = SDPB_MAX; dm.recursion = SDPB_REC_EXPECT; dm.gamma = m.gamma;
            dm.pmf_len = len0.data(); dm.pmf_d = pd.data(); dm.pmf_p = pp.data();
            M = make_model(&dm);
            M.multi = &ml;
            M.tie_tol = m.tie_tolerance;
            td.reset(new TopDown(M));
        } else {
            P.kind = m.kind; P.T = T; P.Q = m.q_bound; P.nD = nD; P.nDt = lens.data();
            P.d1 = m.d1; P.d2 = m.d2; P.p = m.p;
            for (int k = 0; k < 2; k++) { P.price[k] = m.price[k]; P.v[k] = m.vari_cost[k]; P.sal[k] = m.salvage[k]; }
            P.deposit_rate = m.deposit_rate; P.min_inv = m.min_inv; P.max_inv = m.max_inv;
            P.min_cash = m.min_cash; P.max_cash = m.max_cash; P.gamma = m.gamma;
            P.K = m.fixed_cost; P.h = m.hold_cost; P.min_cash_required = m.min_cash_required; P.q = m.state_q;
            rt.reset(new ReachedTopDown(P));
        }
    }
    int ndim() const { return m.kind == SDPB_REACHED_MULTILEAD ? 5 : m.kind == SDPB_REACHED_CASH_ROUNDED ? 2 : 3; }

    St st0(int t, const double* s) const {
        St x; x.t = t; x.x = s[0]; x.x2 = s[1]; x.q1 = s[2]; x.q2 = s[3]; x.w = s[4];
        return x;
    }
    RKey rkey(int t, const double* s) const {
        return m.kind == SDPB_REACHED_CASH_ROUNDED ? RKey{t, s[0], 0.0, s[1]} : RKey{t, s[0], s[1], s[2]};
    }
    double value(const RKey& k) {
        return m.kind == SDPB_REACHED_MULTI_XR ? rt->xr_value(k) : m.kind == SDPB_REACHED_MULTI_YR ? rt->yr_value(k) : rt->cct_value(k);
    }
    // getExpectedValue on an API-order state of period t
    double get(int t, const double* s) { return m.kind == SDPB_REACHED_MULTILEAD ? td->getExpectedValue(st0(t, s)) : value(rkey(t, s)); }

    // |listed actions| of a memo state (MultiProductLeadtime.java:150-158, MultiItemCashXR.java, MultiItemYR.java:104-108,
    // CashConstraintTest.java:76-80)
    double listed(const RKey& s) const {
        if (m.kind == SDPB_REACHED_MULTI_XR) return (double)P.Q * P.Q;
        if (m.kind == SDPB_REACHED_CASH_ROUNDED) {
            const double maxQ = (int)jmin((double)(P.Q - 1), jmax(0, (s.c - P.min_cash_required - P.K) / P.v[0]));
            return (double)((int)maxQ + 1);
        }
        const int miny1 = (int)s.x1, miny2 = (int)s.x2;
        const double iniRf = s.c + P.v[0] * s.x1 + P.v[1] * s.x2;
        double c = 0;
        for (double i = miny1; i < miny1 + P.Q; i = i + 1)
            for (double j = miny2; j < miny2 + P.Q; j = j + 1)
                if (P.v[0] * i + P.v[1] * j < iniRf + 0.1) c++;
        return c;
    }

    // rows [t, state dims (API order)..., a1, a2, V] in map order (at most max_rows); evals derived from the memo
    int64_t rows(double* out, int64_t max_rows, double* evals) {
        const int w = ndim() + 4;
        int64_t r = 0;
        double ev = 0;
        if (m.kind == SDPB_REACHED_MULTILEAD) {
            const int Q = m.q_bound;
            for (auto& kv : td->cacheActions) {
                const St& s = kv.first;
                ev += (double)Q * Q * lens[s.t - 1];
                if (out && r < max_rows) {
                    double* row = out + (size_t)r * w;
                    const int a = (int)kv.second;
                    const double vals[] = {(double)s.t, s.x, s.x2, s.q1, s.q2, s.w, (double)(a / Q), (double)(a % Q),
                                           td->cacheValues.at(s)};
                    std::copy(vals, vals + w, row);
                }
                r++;
            }
        } else {
            for (auto& kv : rt->actions) {
                const RKey& s = kv.first;
                ev += listed(s) * lens[s.t - 1];
                if (out && r < max_rows) {
                    double* row = out + (size_t)r * w;
                    int c = 0;
                    row[c++] = s.t;
                    row[c++] = s.x1;
                    if (m.kind != SDPB_REACHED_CASH_ROUNDED) row[c++] = s.x2;
                    row[c++] = s.c;
                    row[c++] = kv.second.first;
                    row[c++] = kv.second.second;
                    row[c++] = rt->values.at(s);
                }
                r++;
            }
        }
        if (evals) *evals = ev;
        return r;
    }

    // one roll-out (CashSimulation.java:85-118 over this kind's lambdas): getExpectedValue, getAction, the immediate
    // value with d = Math.round(sample), the discounted sum, the transition; kind 2: boundFinalCash after period T
    double path(const double* init, const double* smp /* T * nd */, double discount) {
        const int T = m.T, nd = m.kind == SDPB_REACHED_CASH_ROUNDED ? 1 : 2;
        double sum = 0;
        if (m.kind == SDPB_REACHED_MULTILEAD) {
            St state = st0(1, init);
            const int Q = m.q_bound;
            for (int t = 1; t <= T; t++) {
                td->getExpectedValue(state);
                const int a = (int)td->cacheActions.at(state), a1 = a / Q, a2 = a % Q;
                const int d1 = (int)jround(smp[(t - 1) * nd]), d2 = (int)jround(smp[(t - 1) * nd + 1]);
                sum += std::pow(discount, (double)(t - 1)) * multi_immediate(M, state, a1, a2, d1, d2);
                if (t < T) state = multi_transition(M, state, a1, a2, d1, d2);
            }
            return sum;
        }
        RKey state = rkey(1, init);
        for (int t = 1; t <= T; t++) {
            value(state);
            const std::pair<double, double> a = rt->actions.at(state);
            const double d1 = (double)jround(smp[(t - 1) * nd]), d2 = nd > 1 ? (double)jround(smp[(t - 1) * nd + 1]) : 0.0;
            if (m.kind == SDPB_REACHED_MULTI_YR) {
                const double iniR = state.c + P.v[0] * state.x1 + P.v[1] * state.x2;
                state = rt->yr_transition(state.t, a.first, a.second, iniR, d1, d2);
                if (t == T) sum = rt->yr_value(state);  // boundFinalCash of the state of period T + 1
                continue;
            }
            const double c = m.kind == SDPB_REACHED_MULTI_XR ? rt->xr_immediate(state, a.first, a.second, d1, d2)
                                                             : rt->cct_immediate(state, a.first, d1);
            sum += std::pow(discount, (double)(t - 1)) * c;
            if (t < T)
                state = m.kind == SDPB_REACHED_MULTI_XR ? rt->xr_transition(state, a.first, a.second, d1, d2)
                                                        : rt->cct_transition(state, a.first, d1);
        }
        return sum;
    }
};

}  // namespace

extern "C" {

// getExpectedValue on n API-order states that carry their own period (periods[i]), in call order, on one memo.
// Returns the number of memo states (-1 when kind 0's periods do not share one demand table); rows of ndim + 4 doubles
// [t, state..., a1, a2, V] in map order; values[i] = the i-th call's value; evals = sum over the memo of
// |listed actions| * D_t.
int64_t oracle_reached_at(const sdpb_reached_model* m, const int* periods, const double* states, int n, double* rows,
                          int64_t max_rows, double* values, double* evals) {
    try {
        Memo memo(*m);
        for (int i = 0; i < n; i++) {
            const double v = memo.get(periods[i], states + (size_t)i * memo.ndim());
            if (values) values[i] = v;
        }
        return memo.rows(rows, max_rows, evals);
    } catch (const std::exception&) {
        return -1;
    }
}

// The roll-out loop over one memo, path after path: values[i] = path i's value (samples: n * T * nd, nd = 2 for kinds
// 0-2, 1 for kind 3).  Returns the number of memo states afterwards, rows and evals as oracle_reached_at.
int64_t oracle_reached_simulate(const sdpb_reached_model* m, const double* init_state, const double* samples, int n,
                                double discount, double* values, double* rows, int64_t max_rows, double* evals) {
    try {
        Memo memo(*m);
        const size_t stride = (size_t)m->T * (m->kind == SDPB_REACHED_CASH_ROUNDED ? 1 : 2);
        for (int i = 0; i < n; i++) values[i] = memo.path(init_state, samples + (size_t)i * stride, discount);
        return memo.rows(rows, max_rows, evals);
    } catch (const std::exception&) {
        return -1;
    }
}

}  // extern "C"
