"""sdpb_topdown_*: any single-product model solved over the states its top-down recursion reaches.

Every GPU comparison is bit for bit (==) against oracle_topdown, the literal memoised recursion over real-valued
states, and, where the dense engine can answer the same question, against the dense engine too."""
from __future__ import annotations

import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _in_scope(spec):
    return not (spec.two_product or spec.staff or spec.terminal_value is not None)


IN_SCOPE = [c for c in cases.ALL if _in_scope(c()[0])]


def _options(S, **kw):
    o = S.abi.SdpbTopdownOptions()
    o.struct_size = C.sizeof(S.abi.SdpbTopdownOptions)
    o.device = -1
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def _solve_rc(S, spec, init, opt=None):
    lib = S.abi.load()
    st = np.ascontiguousarray(np.atleast_2d(np.asarray(init, dtype=np.float64)))
    h = C.c_void_p()
    rc = lib.sdpb_topdown_solve(C.byref(spec.to_struct()), opt, st.ctypes.data_as(C.POINTER(C.c_double)),
                                st.shape[0], C.byref(h))
    if rc == 0:
        lib.sdpb_topdown_destroy(h)
    return rc, lib.sdpb_topdown_last_error(None).decode()


# ---- no GPU needed ----------------------------------------------------------------------------------------------------
def test_argument_errors_need_no_gpu(S):
    import torch
    A = S.abi
    for case in (cases.case_M2_small, cases.case_W_small, cases.case_A_terminal):
        spec, init = case()
        rc, msg = _solve_rc(S, spec, init)
        assert rc == A.SDPB_ERR_ARG, (spec.name, msg)
    spec, init = cases.case_A_small()
    m = spec.to_struct()
    m.struct_size = 12
    st = np.asarray(init, dtype=np.float64)
    h = C.c_void_p()
    lib = A.load()
    assert lib.sdpb_topdown_solve(C.byref(m), None, st.ctypes.data_as(C.POINTER(C.c_double)), 1, C.byref(h)) == A.SDPB_ERR_ARG
    bad = _options(S)
    bad.struct_size = 8
    assert _solve_rc(S, spec, init, C.byref(bad))[0] == A.SDPB_ERR_ARG
    assert _solve_rc(S, spec, init, C.byref(_options(S, scratch_bytes=-1)))[0] == A.SDPB_ERR_ARG
    # a valid model: the step need not be a power of two and the state need not be on a grid
    off = S.inventory_model(S.poisson_pmf([3, 3]), max_order=5, inv_min=-5, inv_max=5, step=0.3)
    rc, _ = _solve_rc(S, off, [[2.5]])
    assert rc == (A.SDPB_OK if torch.cuda.is_available() else A.SDPB_ERR_NO_DEVICE)


def test_options_struct_matches_layout_table(S):
    lay = {}
    for line in open(os.path.join(ROOT, "java", "LAYOUT.txt")).read().splitlines():
        if line and not line.startswith("#"):
            name, off, size = line.split()
            lay[name] = (int(off), int(size))
    cls = S.abi.SdpbTopdownOptions
    assert lay["sdpb_topdown_options.sizeof"][0] == C.sizeof(cls)
    assert [k.split(".")[1] for k in lay if k.startswith("sdpb_topdown_options.") and not k.endswith(".sizeof")] == \
        [f for f, _ in cls._fields_]
    for fname, _ in cls._fields_:
        f = getattr(cls, fname)
        assert lay[f"sdpb_topdown_options.{fname}"] == (f.offset, f.size), fname


def test_cpp_wrapper_compiles(tmp_path):
    src = tmp_path / "td.cpp"
    src.write_text('''#include "sdpb200.hpp"
using namespace sdpb200;
int main() {
    const Pmf pmf = GetPmf({PoissonDist(3.0), PoissonDist(3.0)}, 0.999, 1.0).getpmf();
    const Model m = Model::inventory(OptDirection::MIN, pmf, 10, 1, 1, 5, 3, -5, 5, 0.3);
    try {
        TopDown td(m, {{2.5}});
        TopDownRecursion rec(m);
        const double v = rec.getExpectedValue(State{1, 2.5});
        const double q = rec.getAction(State{1, 2.5});
        const bool ok = v == td.value(1, {2.5}) && q >= 0 && td.optTable().size() == td.nStates(1) + td.nStates(2);
        return ok ? 0 : 1;
    } catch (const SdpbError& e) {
        return e.code == SDPB_ERR_NO_DEVICE ? 3 : 2;
    }
}
''')
    exe = tmp_path / "td"
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    "-o", str(exe), "-L", os.path.join(ROOT, "stochastic-inventory_b200"), "-lsdpb200",
                    "-Wl,-rpath," + os.path.join(ROOT, "stochastic-inventory_b200")], check=True)
    import torch
    rc = subprocess.run([str(exe)]).returncode
    assert rc == (0 if torch.cuda.is_available() else 3)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _check_vs_oracle(S, oracle, spec, init, **kw):
    """Rows, values and the evaluation count of the engine == oracle_topdown's; returns the engine."""
    rows, iv, ev = oracle.topdown(spec, init)
    td = S.TopDown(spec, init, **kw)
    nd = spec.ndim
    tab = td.opt_table()
    assert tab.shape == (len(rows), nd + 2), (spec.name, tab.shape, rows.shape)
    assert np.array_equal(tab[:, :nd + 1], rows[:, :nd + 1]), spec.name
    assert np.array_equal(tab[:, -1], rows[:, -2]), spec.name
    assert td.stats()["evals"] == ev, spec.name
    assert td.n_states() == [int((rows[:, 0] == t).sum()) for t in range(1, spec.T + 1)]
    for t in range(1, spec.T + 1):
        sel = rows[rows[:, 0] == t]
        v, q = td.value(t, sel[:, 1:1 + nd])
        assert np.array_equal(v, sel[:, -1]) and np.array_equal(q, sel[:, -2]), (spec.name, t)
    v, _ = td.value(1, init)
    assert np.array_equal(v, iv)
    return td, rows


@pytest.mark.gpu
@pytest.mark.parametrize("case", IN_SCOPE, ids=lambda f: f.__name__[5:])
def test_cases_match_oracle_and_dense(case, S, oracle):
    spec, init = case()
    td, rows = _check_vs_oracle(S, oracle, spec, init)
    dense = S.Solver(spec).solve()
    try:
        dense.reach(init)
    except S.SdpbError:
        return  # the dense grid cannot answer this model from these states (sdpb_reach says why)
    assert np.array_equal(dense.opt_table(), td.opt_table())
    for t in range(1, spec.T + 1):
        sel = rows[rows[:, 0] == t, 1:1 + spec.ndim]
        assert np.array_equal(dense.value(t, sel)[0], td.value(t, sel)[0])


def _off_grid_models(S):
    A = S.abi
    pm = cases.pmf([4, 6, 5])
    half = [np.array([[0.5, 0.25], [1.5, 0.5], [3.0, 0.25]])] * 3
    yield S.inventory_model(pm, fixed_cost=10, vari_cost=1, hold_cost=1, penalty_cost=5, max_order=12, inv_min=-20,
                            inv_max=20, step=0.3, name="step0.3"), [[0.0]]
    yield S.inventory_model(half, fixed_cost=3, vari_cost=0, hold_cost=1, penalty_cost=4, max_order=6, inv_min=-10,
                            inv_max=10, name="half_demands"), [[0.0]]
    yield S.inventory_model(pm, fixed_cost=10, vari_cost=1, hold_cost=1, penalty_cost=5, max_order=10, inv_min=-20,
                            inv_max=20, name="init2.5"), [[2.5]]
    cash = S.cash_constraint_model(cases.pmf([3, 4, 3]), price=5, vari_cost=1, fixed_cost=2, hold_cost=0.5, salvage=0.5,
                                   overhead=1, max_order=8, inv_min=0, inv_max=30, cash_min=0, cash_max=80,
                                   quantiser=A.Q_LONGDIV, q_mul=1.0, q_div=1.0, name="cash33.3")
    yield cash, [[0.0, 33.3]]
    import copy
    frac = copy.copy(cash)
    frac.quantiser, frac.q_mul, frac.q_div, frac.name = A.Q_DIV, 10.0, 10.0, "cash33.33_qdiv"
    yield frac, [[1.0, 33.33]]
    yield S.leadtime_model(cases.pmf([4] * 3), fixed_cost=0, vari_cost=1, hold_cost=2, penalty_cost=10, max_order=12,
                           inv_min=-8, inv_max=20, lead_time=1, clamp=False, name="unclamped_lead1"), [[0.0, 0.0]]
    yield S.cash_survival_model(cases.pmf([5, 6, 5]), price_t=[5.0] * 3, vari_cost_t=[1.0] * 3, overhead_t=[3.0] * 3, fixed_cost=4, max_order=8, inv_min=0,
                                inv_max=20, cash_min=-30, cash_max=60, name="survival_bankrupt"), [[0.0, 6.5]]
    yield S.cash_overdraft_model(cases.pmf([3, 4, 3]), price=6, vari_cost=2, fixed_cost=3, max_order=6, inv_min=0,
                                 inv_max=20, cash_min=-40, cash_max=60, r0=0.01, r2=0.1, r3=0.3, od_limit=20,
                                 name="overdraft_off_grid"), [[1.0, 7.7]]
    lost = copy.copy(cash)
    lost.flags |= A.F_LOST_SALES
    lost.name = "cash_lost_sales"
    yield lost, [[0.0, 12.4]]
    yield S.inventory_model(pm, fixed_cost=10, vari_cost=1, hold_cost=1, penalty_cost=5, max_order=10, inv_min=-20,
                            inv_max=20, step=0.7, name="several_roots"), [[0.0], [2.5], [-1.3], [2.5]]


@pytest.mark.gpu
def test_models_the_dense_engine_refuses(S, oracle):
    seen_bankrupt = False
    for spec, init in _off_grid_models(S):
        td, rows = _check_vs_oracle(S, oracle, spec, init)
        if spec.name == "survival_bankrupt":
            # the engine must not visit a bankrupt successor: every reached state of period > 1 has cash >= 0, while
            # some (state, action, demand) of the model does end below 0 (its values are < 1)
            assert (rows[rows[:, 0] > 1, 2] >= 0).all()
            seen_bankrupt = (rows[:, -1] < 1).any()
    assert seen_bankrupt


@pytest.mark.gpu
def test_xr_capped_action_sets(S, oracle):
    spec, init = cases.case_XR_small()
    with pytest.raises(S.SdpbError) as e:
        S.TopDown(spec, init, allow=0)
    assert e.value.code == S.abi.SDPB_ERR_OFFGRID
    td, _ = _check_vs_oracle(S, oracle, spec, init, allow=S.ALLOW_CAPPED_ACTIONS)
    assert td.stats()["capped_action_sets"] > 0


@pytest.mark.gpu
def test_chunked_expansion_matches_one_pass(S, oracle):
    """A scratch budget far below one period's candidates: many chunks, the same states and values as one pass.  A
    budget below what a period's reached states need: SDPB_ERR_NOMEM naming the period."""
    A = S.abi
    spec = S.cash_constraint_model(cases.pmf([8, 10, 8, 9]), price=5, vari_cost=1, fixed_cost=2, hold_cost=0.5,
                                   salvage=0.5, overhead=1, max_order=20, inv_min=0, inv_max=60, cash_min=0,
                                   cash_max=300, quantiser=A.Q_LONGDIV, q_mul=1.0, q_div=1.0, name="chunked")
    init = [[0.0, 50.5]]
    whole, rows = _check_vs_oracle(S, oracle, spec, init)
    n = whole.n_states()
    # room for twice the largest frontier plus 4000 keys in each of the three buffers, and 4 MiB for the sort's
    # temporary storage: at most ~62000 candidates per chunk
    budget = 3 * 32 * (2 * max(n) + 4000) + (4 << 20)
    sel = rows[rows[:, 0] == 3]
    cand = sum(oracle.n_actions(spec, 3, r[1:3]) for r in sel) * len(spec.pmf[2])
    assert cand > 10 * budget // (3 * 32)      # period 4 is expanded in ten chunks or more
    small = S.TopDown(spec, init, scratch_bytes=budget)
    assert np.array_equal(small.opt_table(), whole.opt_table())
    assert small.stats()["evals"] == whole.stats()["evals"]
    for t in range(1, spec.T + 1):
        st = rows[rows[:, 0] == t, 1:3]
        assert np.array_equal(small.value(t, st)[0], whole.value(t, st)[0])
    for tight in (3 * 32 * max(n), 3 * 32 * 2000):
        with pytest.raises(S.SdpbError) as e:
            S.TopDown(spec, init, scratch_bytes=tight)
        assert e.value.code == A.SDPB_ERR_NOMEM and "period" in str(e.value)


@pytest.mark.gpu
def test_survival_root_whose_successors_all_go_bankrupt(S, oracle):
    """Every successor of the root has negative cash, so the survival recursion visits nothing after period 1: the
    later periods are empty and the root is worth 0 with action 0, as in the reference (solve_state never recurses)."""
    spec = S.cash_survival_model(cases.pmf([5, 6, 5]), max_order=8, inv_min=0, inv_max=20)   # overhead 100
    for init in ([[0.0, 0.0]], [[0.0, 0.0], [0.0, -29.0]], [[0.0, 0.0], [3.0, 150.0]]):
        td, rows = _check_vs_oracle(S, oracle, spec, init)
        if len(init) == 2 and init[1][1] < 0:
            assert td.n_states()[1:] == [0, 0]
    assert S.RiskRecursion(spec, topdown=True).getSurvProb(S.RiskState(1, 0.0, 0.0)) == 0.0
    with pytest.raises(KeyError):
        S.RiskRecursion(spec, topdown=True).getAction(S.RiskState(2, 0.0, 0.0))


@pytest.mark.gpu
def test_queries(S):
    spec, init = cases.case_A_small()
    td = S.TopDown(spec, init)
    with pytest.raises(S.SdpbError) as e:
        td.value(2, [[1e6]])
    assert e.value.code == S.abi.SDPB_ERR_UNSOLVED
    for bad in (0, spec.T + 1):
        with pytest.raises(S.SdpbError) as e:
            td.value(bad, init)
        assert e.value.code == S.abi.SDPB_ERR_ARG
    td.close()


@pytest.mark.gpu
def test_facades(S, oracle):
    pm = cases.pmf([4, 6, 5])
    inv = S.inventory_model(pm, fixed_cost=10, vari_cost=1, hold_cost=1, penalty_cost=5, max_order=10, inv_min=-20,
                            inv_max=20, step=0.5)
    rec = S.Recursion(inv, topdown=True)
    rows, iv, _ = oracle.topdown(inv, [[2.25]])
    assert rec.getExpectedValue(S.State(1, 2.25)) == iv[0]
    assert np.array_equal(rec.getOptTable(), rows[:, :-1])
    assert rec.getAction(S.State(1, 2.25)) == rows[(rows[:, 0] == 1) & (rows[:, 1] == 2.25), -2][0]
    with pytest.raises(KeyError):
        rec.getAction(S.State(2, 1e6))
    # a second root re-solves with both
    iv2 = oracle.topdown(inv, [[2.25], [-0.75]])[1]
    assert rec.getExpectedValue(S.State(1, -0.75)) == iv2[1]
    assert len(rec.getCacheActions()) == len(oracle.topdown(inv, [[2.25], [-0.75]])[0])

    cash = S.cash_constraint_model(cases.pmf([3, 4, 3]), price=5, vari_cost=1, fixed_cost=2, hold_cost=0.5, salvage=0.5,
                                   overhead=1, max_order=8, inv_min=0, inv_max=30, cash_min=0, cash_max=80)
    assert S.CashRecursion(cash, topdown=True).getExpectedValue(S.CashState(1, 0.5, 33.3)) == \
        oracle.topdown(cash, [[0.5, 33.3]])[1][0]
    lead = S.leadtime_model(cases.pmf([4] * 3), fixed_cost=0, vari_cost=1, hold_cost=2, penalty_cost=10, max_order=12,
                            inv_min=-8, inv_max=20, lead_time=1, clamp=False)
    assert S.LeadtimeRecursion(lead, topdown=True).getExpectedValue(S.LeadtimeState(1, 0.5, 1.0)) == \
        oracle.topdown(lead, [[0.5, 1.0]])[1][0]
    surv = S.cash_survival_model(cases.pmf([5, 6, 5]), price_t=[5.0] * 3, vari_cost_t=[1.0] * 3, overhead_t=[3.0] * 3, fixed_cost=4, max_order=8, inv_min=0,
                                 inv_max=20, cash_min=-30, cash_max=60)
    assert S.RiskRecursion(surv, topdown=True).getSurvProb(S.RiskState(1, 0.0, 6.5)) == \
        oracle.topdown(surv, [[0.0, 6.5]])[1][0]


def _random_model(S, family, rng):
    A = S.abi
    T = rng.randint(2, 4)
    step = rng.choice([0.3, 0.7, 1.0, 1.5, 2.5])
    means = [rng.uniform(1, 6) for _ in range(T)]
    pm = [np.column_stack([np.round(r[:, 0] * rng.choice([0.5, 0.7, 1.0]), 3), r[:, 1]]) for r in cases.pmf(means)]
    maxq = rng.randint(2, 9)
    x0 = round(rng.uniform(-3, 6), 2)
    w0 = round(rng.uniform(0, 40), 2)
    if family == "backorder":
        spec = S.inventory_model(pm, fixed_cost=rng.choice([0, 5, 12.5]), vari_cost=rng.choice([0, 1, 0.5]),
                                 hold_cost=1, penalty_cost=rng.choice([4, 9.5]), max_order=maxq, inv_min=-30, inv_max=30,
                                 step=step)
        spec.flags = rng.choice([A.F_CLAMP_INV, 0, A.F_CLAMP_INV | A.F_LOST_SALES, A.F_CLAMP_INV | A.F_GY_MODE])
        return spec, [[x0]]
    if family == "leadtime":
        L = rng.choice([1, 2])
        spec = S.leadtime_model(pm, fixed_cost=rng.choice([0, 3]), vari_cost=1, hold_cost=2, penalty_cost=10,
                                max_order=min(maxq, 5), inv_min=-25, inv_max=25, lead_time=L, clamp=rng.random() < 0.5,
                                step=step)
        if rng.random() < 0.3:
            spec.flags |= A.F_NO_ORDER_LAST
        return spec, [[x0] + [round(rng.uniform(0, 4), 1)] * L]
    kw = dict(max_order=maxq, inv_min=0, inv_max=25, cash_min=rng.choice([0, -20]), cash_max=rng.choice([60, 90]))
    if family == "deposit":
        spec = S.cash_constraint_model(pm, price=rng.choice([4, 5.5]), vari_cost=1, fixed_cost=rng.choice([0, 2]),
                                       hold_cost=0.5, salvage=0.5, overhead=rng.choice([0, 1.5]), **kw)
        if rng.random() < 0.5:
            spec.flags |= A.F_CASH_LIMITED_ACTIONS
        spec.quantiser, spec.q_mul, spec.q_div = rng.choice([(A.Q_LONGDIV, 1.0, 1.0), (A.Q_DIV, 10.0, 10.0)])
    elif family == "overdraft":
        spec = S.cash_overdraft_model(pm, price=6, vari_cost=2, fixed_cost=rng.choice([0, 3]), r0=0.01,
                                      r2=0.1, r3=0.3, od_limit=20, **kw)
    elif family == "survival":
        spec = S.cash_survival_model(pm, price_t=[3.0] * T, vari_cost_t=[2.0] * T, overhead_t=[1.0] * T, fixed_cost=rng.choice([0, 4]), **kw)
    elif family == "xr":
        spec = S.cash_xr_model(pm, price=5, vari_cost=1, fixed_cost=rng.choice([0, 2]), **kw)
        spec.allow, spec.step = A.ALLOW_CAPPED_ACTIONS, step
        return spec, [[abs(x0), w0 + abs(x0)]]
    elif family == "od_limit":
        spec = S.cash_overdraft_limit_model(pm, price=5, vari_cost=1, fixed_cost=2, hold_cost=0.5,
                                            interest_rate=0.1, **kw)
    elif family == "od_testing":
        spec = S.cash_overdraft_testing_model(pm, price=5, vari_cost=1, fixed_cost=2, hold_cost=0.5,
                                              interest_rate=0.1, **kw)
    else:
        spec = S.cash_loan_model(pm, price=5, vari_cost=1, hold_cost=0.5, salvage=0.5, loan_rate=0.1, **kw)
    spec.step = step
    if rng.random() < 0.5:
        spec.flags |= A.F_LOST_SALES
    return spec, [[abs(x0), w0]]


FAMILIES = ["backorder", "leadtime", "deposit", "overdraft", "survival", "xr", "od_limit", "od_testing", "loan"]


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_seeded_fuzz(family, S, oracle):
    rng = random.Random(20261020 + FAMILIES.index(family))
    for _ in range(20):
        spec, init = _random_model(S, family, rng)
        _check_vs_oracle(S, oracle, spec, init)
