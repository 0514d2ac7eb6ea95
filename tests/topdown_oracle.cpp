// CPU references for sdpb_topdown_extend and sdpb_topdown_simulate (test infrastructure; never linked into
// libsdpb200.so).  The oracle's own TopDown, solve_state, immediate and transition are used unchanged: this file
// includes oracle/sdp_oracle.cpp and adds two entry points that drive one memoised TopDown in a new order.
// Built by tests/topdown_oracle.py with the oracle's flags (-ffp-contract=off: Java never fuses multiply-add).
#include "../oracle/sdp_oracle.cpp"

namespace {

// The memo of `td` as oracle_topdown writes it: rows of (ndim + 3) doubles [t, state dims..., Q*, V], at most max_rows.
int64_t memo_rows(const Grid& G, TopDown& td, double* rows, int64_t max_rows) {
    const int64_t n = (int64_t)td.cacheActions.size();
    if (!rows) return n;
    const int w = G.ndim() + 3;
    int64_t r = 0;
    for (auto& kv : td.cacheActions) {
        if (r >= max_rows) break;
        double* row = rows + (size_t)r * w;
        row[0] = kv.first.t;
        G.to_api(kv.first, row + 1);
        row[1 + G.ndim()] = kv.second;
        row[2 + G.ndim()] = td.cacheValues[kv.first];
        r++;
    }
    return n;
}

}  // namespace

extern "C" {

// TopDown::getExpectedValue on `n` states that carry their own period (periods[i], API-order states), in call order,
// all on one memo.  Returns the number of memoised states; rows as oracle_topdown; values[i] = the i-th call's value.
int64_t oracle_topdown_at(const sdpb_model* m, const int* periods, const double* states, int n, double* rows,
                          int64_t max_rows, double* values, double* evals) {
    Model M = make_model(m);
    Grid G(M);
    TopDown td(M);
    for (int i = 0; i < n; i++) {
        const double v = td.getExpectedValue(G.from_api(periods[i], states + (size_t)i * G.ndim()));
        if (values) values[i] = v;
    }
    if (evals) *evals = td.evals;
    return memo_rows(G, td, rows, max_rows);
}

// Simulation.java:59-70 (CashSimulation.java:100-111) literally, over one TopDown: at every step
// getExpectedValue(state) -- which solves and memoises a state not seen yet -- then cacheActions[state], then the
// immediate value and the transition with the rounded sample.  values[i] = path i's sum; returns the number of memoised
// states afterwards, rows as oracle_topdown.
int64_t oracle_topdown_simulate(const sdpb_model* m, const double* init_state, const double* samples, int n,
                                double discount, double* values, double* rows, int64_t max_rows, double* evals) {
    Model M = make_model(m);
    Grid G(M);
    TopDown td(M);
    const int T = m->T;
    for (int i = 0; i < n; i++) {
        double sum = 0;
        St state = G.from_api(1, init_state);
        for (int t = 0; t < T; t++) {
            td.getExpectedValue(state);
            const double optQ = td.cacheActions.at(state);
            const double randomDemand = (double)jround(samples[(size_t)i * T + t]);
            const double thisValue = immediate(M, state, optQ, randomDemand);
            sum += std::pow(discount, (double)t) * thisValue;
            state = transition(M, state, optQ, randomDemand);
        }
        values[i] = sum;
    }
    if (evals) *evals = td.evals;
    return memo_rows(G, td, rows, max_rows);
}

}  // extern "C"
