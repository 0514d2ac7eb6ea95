"""sdpb_topdown_extend / sdpb_topdown_simulate: a top-down solve extended with states of any period, and the policy
rolled out over sample paths with the reference's lazy getExpectedValue at every step (Simulation.java:62).

Every GPU comparison is bit for bit (==) against the oracle's literal memoised recursion (tests/topdown_oracle.py):
oracle_topdown_at for the same getExpectedValue calls, oracle_topdown_simulate for the same roll-out."""
from __future__ import annotations

import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import cases
import topdown_oracle as TO
from test_topdown import FAMILIES, IN_SCOPE, _off_grid_models, _random_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp = C.POINTER(C.c_double)


def _arr(a):
    return np.ascontiguousarray(np.atleast_2d(np.asarray(a, dtype=np.float64)))


# ---- no GPU needed ----------------------------------------------------------------------------------------------------
def test_null_handle_is_an_argument_error(S):
    lib = S.abi.load()
    st, sm, out = _arr([[0.0]]), _arr([[1.0, 2.0]]), np.empty(1)
    assert lib.sdpb_topdown_extend(None, 1, st.ctypes.data_as(_dp), 1) == S.abi.SDPB_ERR_ARG
    assert lib.sdpb_topdown_simulate(None, st.ctypes.data_as(_dp), sm.ctypes.data_as(_dp), 1, 1.0,
                                     out.ctypes.data_as(_dp)) == S.abi.SDPB_ERR_ARG


def test_cpp_extend_and_simulate_compile(tmp_path):
    src = tmp_path / "td.cpp"
    src.write_text('''#include "sdpb200.hpp"
using namespace sdpb200;
int main() {
    const Pmf pmf = GetPmf({PoissonDist(3.0), PoissonDist(3.0)}, 0.999, 1.0).getpmf();
    const Model m = Model::inventory(OptDirection::MIN, pmf, 10, 1, 1, 5, 3, -5, 5, 0.3);
    try {
        TopDown td(m, {{2.5}});
        const sdpb_stats s0 = td.stats();
        td.extend(2, {{1.15}, {-0.35}});
        const std::vector<double> v = td.simulate({2.5}, {{2.6, 9.4}, {0.0, 3.0}, {-0.4, 1.49}}, 0.9);
        TopDownRecursion rec(m);
        const double a = rec.getExpectedValue(State{1, 2.5});
        const double b = rec.getExpectedValue(State{1, 0.7});
        const bool ok = v.size() == 3 && a == td.value(1, {2.5}) && b == rec.engine().value(1, {0.7}) &&
                        td.stats().evals > s0.evals && td.nStates(2) >= 2;
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
def _snapshot(td):
    return td.opt_table(), td.n_states(), td.stats()["evals"], td.stats()["capped_action_sets"]


def _assert_memo(S, td, spec, rows, ev, what):
    """opt_table, the value at every reached state and evals == the oracle's memo rows [t, state..., Q, V]."""
    nd = spec.ndim
    tab = td.opt_table()
    assert tab.shape == (len(rows), nd + 2), (what, tab.shape, rows.shape)
    assert np.array_equal(tab[:, :nd + 1], rows[:, :nd + 1]), what
    assert np.array_equal(tab[:, -1], rows[:, -2]), what
    assert td.stats()["evals"] == ev, what
    for t in range(1, spec.T + 1):
        sel = rows[rows[:, 0] == t]
        if len(sel):
            v, q = td.value(t, sel[:, 1:1 + nd])
            assert np.array_equal(v, sel[:, -1]) and np.array_equal(q, sel[:, -2]), (what, t)


def _unreached(rows, spec, t, k=3):
    """Up to k states of period t that no root reaches: reached ones with their inventory moved off every grid."""
    sel = rows[rows[:, 0] == t, 1:1 + spec.ndim][:k].copy()
    sel[:, 0] += 0.3712
    return sel


def _extension_steps(S, spec, init):
    """solve; extend with reached states (no-op); extend with unreached states of periods 2..T; extend with a new
    period-1 root.  After each step the handle == oracle_topdown_at on the same calls."""
    init = [list(r) for r in init]
    calls = [(1, r) for r in init]
    td = S.TopDown(spec, init)
    rows, _, ev = TO.topdown_at(spec, [c[0] for c in calls], [c[1] for c in calls])
    _assert_memo(S, td, spec, rows, ev, (spec.name, "solve"))
    n0, ev0 = td.n_states(), td.stats()["evals"]
    for t in range(2, spec.T + 1):
        sel = rows[rows[:, 0] == t, 1:1 + spec.ndim][:4]
        if len(sel):
            td.extend(t, sel)
            calls += [(t, list(r)) for r in sel]
    assert td.n_states() == n0 and td.stats()["evals"] == ev0, spec.name
    grew = False
    for t in range(2, spec.T + 1):
        new = _unreached(rows, spec, t)
        if len(new):
            td.extend(t, new)
            calls += [(t, list(r)) for r in new]
            grew = True
    want, _, ev = TO.topdown_at(spec, [c[0] for c in calls], [c[1] for c in calls])
    _assert_memo(S, td, spec, want, ev, (spec.name, "later periods"))
    root = list(init[0])
    root[0] += 1.13
    td.extend(1, [root])
    calls.append((1, root))
    want, vals, ev = TO.topdown_at(spec, [c[0] for c in calls], [c[1] for c in calls])
    _assert_memo(S, td, spec, want, ev, (spec.name, "new root"))
    assert td.value(1, [root])[0][0] == vals[-1]
    return grew and len(want) > len(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("case", IN_SCOPE, ids=lambda f: f.__name__[5:])
def test_extend_matches_oracle(case, S):
    spec, init = case()
    grew = _extension_steps(S, spec, init)
    assert grew or spec.T == 1


@pytest.mark.gpu
def test_extend_off_grid_models_match_oracle(S):
    for spec, init in _off_grid_models(S):
        _extension_steps(S, spec, init)


@pytest.mark.gpu
def test_roots_one_by_one_equal_one_solve(S):
    for spec, init in _off_grid_models(S):
        roots = [list(init[0]), [init[0][0] + 0.9] + list(init[0][1:]), [init[0][0] + 2.45] + list(init[0][1:])]
        whole = S.TopDown(spec, roots)
        one = S.TopDown(spec, roots[:1])
        for r in roots[1:]:
            one.extend(1, [r])
        assert np.array_equal(one.opt_table(), whole.opt_table()), spec.name
        assert one.stats()["evals"] == whole.stats()["evals"], spec.name
        for t in range(1, spec.T + 1):
            st = whole.opt_table()
            st = st[st[:, 0] == t, 1:1 + spec.ndim]
            if len(st):
                assert np.array_equal(one.value(t, st)[0], whole.value(t, st)[0]), (spec.name, t)


@pytest.mark.gpu
def test_failed_extension_leaves_the_handle_as_it_was(S):
    A = S.abi
    # NOMEM: 15000 period-2 roots on distinct off-grid levels fit a buffer, their successors in period 3 do not
    pm = cases.pmf([4, 6, 5])
    spec = S.inventory_model(pm, fixed_cost=10, vari_cost=1, hold_cost=1, penalty_cost=5, max_order=10, inv_min=-500,
                             inv_max=500, step=0.7, name="unclamped")
    spec.flags = 0
    td = S.TopDown(spec, [[0.0]], scratch_bytes=3 * 32 * 20000 + (4 << 20))
    before = _snapshot(td)
    with pytest.raises(S.SdpbError) as e:
        td.extend(2, (np.arange(15000) * 1e-3 + 1e-4)[:, None])
    assert e.value.code == A.SDPB_ERR_NOMEM and "period 3" in str(e.value), str(e.value)
    after = _snapshot(td)
    assert np.array_equal(after[0], before[0]) and after[1:] == before[1:]
    td.extend(2, [[0.35]])  # still usable
    rows, _, ev = TO.topdown_at(spec, [1, 2], [[0.0], [0.35]])
    _assert_memo(S, td, spec, rows, ev, "after NOMEM")

    # OFFGRID: an XR state whose order-up-to range is longer than max_order_idx + 1, without the allow bit
    xr = S.cash_xr_model(cases.pmf([3, 4, 3]), price=5, vari_cost=1, fixed_cost=2, max_order=60, inv_min=0, inv_max=25,
                         cash_min=0, cash_max=20)
    td = S.TopDown(xr, [[2.0, 12.0]], allow=0)
    before = _snapshot(td)
    with pytest.raises(S.SdpbError) as e:
        td.extend(2, [[1.0, 500.0]])
    assert e.value.code == A.SDPB_ERR_OFFGRID
    after = _snapshot(td)
    assert np.array_equal(after[0], before[0]) and after[1:] == before[1:]


@pytest.mark.gpu
def test_argument_errors(S):
    A = S.abi
    lib = A.load()
    spec, init = cases.case_A_small()
    td = S.TopDown(spec, init)
    before = _snapshot(td)
    st = _arr(init)
    for period, n in ((0, 1), (spec.T + 1, 1), (1, -1)):
        assert lib.sdpb_topdown_extend(td.h, period, st.ctypes.data_as(_dp), n) == A.SDPB_ERR_ARG
    assert lib.sdpb_topdown_extend(td.h, 2, st.ctypes.data_as(_dp), 0) == A.SDPB_OK
    for bad in (np.nan, np.inf):
        with pytest.raises(S.SdpbError) as e:
            td.extend(2, [[bad]])
        assert e.value.code == A.SDPB_ERR_ARG
    sm = _arr(np.ones((4, spec.T)))
    out = np.empty(4)
    sim = lib.sdpb_topdown_simulate
    assert sim(td.h, None, sm.ctypes.data_as(_dp), 4, 1.0, out.ctypes.data_as(_dp)) == A.SDPB_ERR_ARG
    assert sim(td.h, st.ctypes.data_as(_dp), None, 4, 1.0, out.ctypes.data_as(_dp)) == A.SDPB_ERR_ARG
    assert sim(td.h, st.ctypes.data_as(_dp), sm.ctypes.data_as(_dp), 4, 1.0, None) == A.SDPB_ERR_ARG
    assert sim(td.h, st.ctypes.data_as(_dp), sm.ctypes.data_as(_dp), 0, 1.0, out.ctypes.data_as(_dp)) == A.SDPB_ERR_ARG
    nan_sm = sm.copy()
    nan_sm[2, 1] = np.nan
    with pytest.raises(S.SdpbError) as e:
        td.simulate(init[0], nan_sm)
    assert e.value.code == A.SDPB_ERR_ARG
    with pytest.raises(S.SdpbError) as e:
        td.simulate([np.inf], sm)
    assert e.value.code == A.SDPB_ERR_ARG
    with pytest.raises(ValueError):
        td.simulate(init[0], np.ones((4, spec.T + 1)))
    after = _snapshot(td)
    assert np.array_equal(after[0], before[0]) and after[1:] == before[1:]


def _samples(spec, n, seed):
    rng = np.random.default_rng(seed)
    dmax = max(r[-1, 0] for r in spec.pmf)
    return rng.uniform(-0.4, dmax + 3.0, size=(n, spec.T))  # out-of-support and fractional draws


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_rollout_fuzz_matches_oracle(family, S):
    rng = random.Random(20261021 + FAMILIES.index(family))
    rounds = []
    for k in range(10):
        spec, init = _random_model(S, family, rng)
        samples = _samples(spec, 300, 100 * FAMILIES.index(family) + k)
        for discount in (1.0, 0.9):
            td = S.TopDown(spec, init)
            got = td.simulate(init[0], samples, discount)
            rounds.append(td.stats()["launches"])
            want, rows, ev = TO.topdown_simulate(spec, init[0], samples, discount)
            assert np.array_equal(got, want), (family, k, discount)
            _assert_memo(S, td, spec, rows, ev, (family, k, discount))
    assert max(rounds) >= 2, rounds  # some roll-outs stalled, extended the handle and went on in a second round


@pytest.mark.gpu
@pytest.mark.parametrize("case", [cases.case_A_small, cases.case_B1_fixed, cases.case_B2_small, cases.case_C_rich,
                                  cases.case_C_int, cases.case_D_rich, cases.case_E_small, cases.case_XR_small,
                                  cases.case_DT_small], ids=lambda f: f.__name__[5:])
def test_rollout_matches_dense_rollout(case, S):
    """The clamped cases of the dense roll-out's parity test: there the oracle's dense and top-down roll-outs agree."""
    spec, init = case()
    samples = _samples(spec, 500, 5)
    want = S.Solver(spec).solve().simulate(init[0], samples, spec.gamma)
    got = S.TopDown(spec, init[:1]).simulate(init[0], samples, spec.gamma)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_reference_style_simulation(S):
    """CLSPTesting.java:125-127 with a step the dense engine cannot take: Simulation(distributions, sampleNum,
    recursion) over a top-down recursion."""
    dists = [S.PoissonDist(m) for m in (5, 8, 6)]
    pmf = S.GetPmf(dists, 0.999, 1).getpmf()
    spec = S.inventory_model(pmf, 20, 1, 1, 5, max_order=30, inv_min=-30, inv_max=30, step=0.5)
    recursion = S.Recursion(spec, topdown=True)
    sim = S.Simulation(dists, 2000, recursion)
    samples = S.generate_lh_samples(dists, 2000)
    paths = sim.simulate_paths(S.State(1, 0), samples)
    opt = recursion.getExpectedValue(S.State(1, 0))
    mean = sim.simulateSDPGivenSamplNum(S.State(1, 0), samples)
    assert abs(mean - opt) / opt < 0.05
    want, memo, _ = TO.topdown_simulate(spec, [0.0], samples)
    assert np.array_equal(paths, want)
    assert np.array_equal(recursion.getOptTable(), memo[:, :-1])
    # a period-1 root after the roll-out keeps the simulated states, as the reference's memo does; the memo is the
    # closure of every state asked for, so the oracle's is rebuilt from the roll-out's memo plus the new root
    recursion.getExpectedValue(S.State(1, 3.5))
    rows, _, _ = TO.topdown_at(spec, list(memo[:, 0].astype(int)) + [1], np.vstack([memo[:, 1:2], [[3.5]]]))
    assert np.array_equal(recursion.getOptTable(), rows[:, :-1])
    assert len(recursion.getCacheActions()) == len(rows)

    cash = S.cash_constraint_model(cases.pmf([3, 4, 3]), price=5, vari_cost=1, fixed_cost=2, hold_cost=0.5,
                                   salvage=0.5, overhead=1, max_order=8, inv_min=0, inv_max=30, cash_min=0, cash_max=80)
    csamples = _samples(cash, 1000, 7)
    crec = S.CashRecursion(cash, topdown=True)
    csim = S.CashSimulation([], 1000, crec, discountFactor=0.95)
    got = csim.simulateSDPGivenSamplNum(S.CashState(1, 0.5, 33.3), csamples)
    cvals, _, _ = TO.topdown_simulate(cash, [0.5, 33.3], csamples, 0.95)
    assert got == float(cvals.sum() / len(cvals)) + 33.3
