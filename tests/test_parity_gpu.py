"""GPU parity tests: libsdpb200.so (through the C-ABI) against the CPU oracle, bit for bit.

Values are compared with ==, order quantities with == (the argopt reduction reproduces the
reference's first-wins tie rule, so even exact ties must agree)."""
import ctypes as C

import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu


def _solve_all(S, spec, **kw):
    s = S.Solver(spec, **kw)
    s.solve()
    V = np.empty((spec.T, s.n_states))
    Q = np.empty((spec.T, s.n_states))
    for t in range(1, spec.T + 1):
        V[t - 1], Q[t - 1] = s.period_tables(t)
    return s, V, Q


@pytest.mark.parametrize("case", cases.ALL, ids=lambda f: f.__name__[5:])
def test_generic_kernel_whole_grid(case, S, oracle):
    spec, init = case()
    Vo, Qo, evals, _ = oracle.dense(spec)
    s, V, Q = _solve_all(S, spec, kernel=S.KERNEL_GENERIC)
    assert s.n_states == Vo.shape[1]
    assert np.array_equal(V, Vo)
    assert np.array_equal(Q, Qo)
    st = s.stats()
    assert st["evals"] == evals
    assert st["launches"] == spec.T and st["kernel_used"] == S.KERNEL_GENERIC


@pytest.mark.parametrize("case", cases.ALL, ids=lambda f: f.__name__[5:])
def test_auto_kernel_whole_grid(case, S, oracle):
    """Whatever kernel AUTO picks (tiled where one exists) must give the same bits."""
    spec, init = case()
    Vo, Qo, evals, _ = oracle.dense(spec)
    s, V, Q = _solve_all(S, spec)
    assert np.array_equal(V, Vo)
    assert np.array_equal(Q, Qo)
    assert s.stats()["evals"] == evals


A_CASES = [cases.case_A_small, cases.case_A_max, cases.case_A_gy, cases.case_A_twopoint, cases.case_A_halfstep,
           cases.case_A_sparse_pmf, cases.case_A_degenerate, cases.case_A_one_state]


@pytest.mark.parametrize("case", A_CASES, ids=lambda f: f.__name__[5:])
@pytest.mark.parametrize("kernel", ["tiled", "tiled2"])
def test_both_tiled_variants_whole_grid(case, kernel, S, oracle):
    """bi_inv_tiled (1 level x 8 actions per thread) and bi_inv_tiled2 (4 levels x 4 actions, sliding
    register window), forced on small grids so the action-split / last-CTA merge path runs too."""
    spec, init = case()
    Vo, Qo, evals, _ = oracle.dense(spec)
    k = S.KERNEL_TILED if kernel == "tiled" else S.KERNEL_TILED2
    s, V, Q = _solve_all(S, spec, kernel=k)
    assert np.array_equal(V, Vo)
    assert np.array_equal(Q, Qo)
    used = s.stats()["kernel_used"]
    if kernel == "tiled2" and case is not cases.case_A_twopoint:   # two-point demand is not consecutive
        assert used == S.KERNEL_TILED2
    else:
        assert used == S.KERNEL_TILED


def test_tiled2_wide_cases(S, oracle):
    """Shapes that exercise tile edges of the 1021-state tile: several tiles, D not a multiple of 4,
    action count not a multiple of 4, MAX direction."""
    for (n_inv, max_order, means, direction) in [(2500, 37, [7, 9, 8], S.MIN), (1021 * 2 + 5, 10, [3, 11], S.MAX),
                                                 (1500, 3, [2, 2, 2], S.MIN)]:
        spec = S.inventory_model(S.poisson_pmf(means, 0.999), fixed_cost=12, vari_cost=1, hold_cost=1,
                                 penalty_cost=6, max_order=max_order, inv_min=-(n_inv // 2),
                                 inv_max=n_inv - n_inv // 2 - 1, direction=direction)
        Vo, Qo, _, _ = oracle.dense(spec)
        for k in (S.KERNEL_TILED2, S.KERNEL_TILED):
            s, V, Q = _solve_all(S, spec, kernel=k)
            assert np.array_equal(V, Vo) and np.array_equal(Q, Qo), (n_inv, max_order, k)


LEAD_CASES = [cases.case_B1_ref, cases.case_B1_fixed, cases.case_B2_small, cases.case_E_small]


@pytest.mark.parametrize("case", LEAD_CASES, ids=lambda f: f.__name__[5:])
@pytest.mark.parametrize("kernel", ["auto", "generic"])
def test_dedup_whole_grid(case, kernel, S, oracle):
    """Lead-time models depend on (x, preQ) only through x + preQ; folding those states is exact."""
    spec, init = case()
    Vo, Qo, evals, _ = oracle.dense(spec)
    k = S.KERNEL_AUTO if kernel == "auto" else S.KERNEL_GENERIC
    s, V, Q = _solve_all(S, spec, dedup=True, kernel=k)
    assert np.array_equal(V, Vo)
    assert np.array_equal(Q, Qo)
    st = s.stats()
    assert st["evals"] == evals and 0 < st["evals_executed"] < evals


@pytest.mark.parametrize("case", [cases.case_C_int, cases.case_C_int_K, cases.case_F_small],
                         ids=lambda f: f.__name__[5:])
def test_integer_cash_kernels_whole_grid(case, S, oracle):
    """bi_cash_diag (AUTO) and bi_cash_int (requested) against the oracle."""
    spec, _ = case()
    Vo, Qo, _, _ = oracle.dense(spec)
    for k, used in ((S.KERNEL_AUTO, S.KERNEL_CASH_DIAG), (S.KERNEL_CASH_INT, S.KERNEL_CASH_INT)):
        s, V, Q = _solve_all(S, spec, kernel=k)
        assert s.stats()["kernel_used"] == used, spec.name
        assert np.array_equal(V, Vo) and np.array_equal(Q, Qo), (spec.name, k)


def test_cash_diag_wide_cases(S, oracle):
    """Diagonal-window kernel edges: price larger than the cash tile step, inventory rows not a multiple
    of 8, short and long demand tables (stock-out region dominant / absent), MIN direction, discounting."""
    for (price, v, K, means, inv_max, cash_max, max_order, direction, gamma) in [
            (10, 1, 0, [5, 6, 5], 21, 300, 13, S.MAX, 1.0), (3, 2, 4, [9, 3], 30, 150, 20, S.MAX, 0.9),
            (25, 3, 0, [2, 2, 2], 9, 400, 6, S.MIN, 1.0), (7, 1, 2, [30, 28], 70, 260, 40, S.MAX, 1.0)]:
        spec = S.cash_constraint_model(S.poisson_pmf(means, 0.999), price=price, vari_cost=v, fixed_cost=K,
                                       salvage=0.5, max_order=max_order, inv_min=0, inv_max=inv_max, cash_min=-20,
                                       cash_max=cash_max, quantiser=S.Q_LONGDIV, q_mul=1.0, q_div=1.0, gamma=gamma,
                                       direction=direction)
        Vo, Qo, _, _ = oracle.dense(spec)
        s, V, Q = _solve_all(S, spec)
        assert s.stats()["kernel_used"] == S.KERNEL_CASH_DIAG
        assert np.array_equal(V, Vo) and np.array_equal(Q, Qo), (price, v, K, means)


def test_integer_cash_kernel_is_used(S):
    for case in (cases.case_C_int, cases.case_C_int_K, cases.case_F_small):
        spec, _ = case()
        assert S.Solver(spec).solve().stats()["kernel_used"] == S.KERNEL_CASH_DIAG, spec.name
    # fractional cash grids and the overdraft lambdas: the cash-independent terms are shared across a row of cash levels
    # (bi_cash_tail); the survival recursion keeps the older row kernel, the remaining kinds the generic one
    for case, used in ((cases.case_C_small, S.KERNEL_CASH_TAIL), (cases.case_C_rich, S.KERNEL_CASH_TAIL),
                       (cases.case_D_small, S.KERNEL_CASH_TAIL), (cases.case_D_rich, S.KERNEL_CASH_TAIL),
                       (cases.case_DL_small, S.KERNEL_CASH_TAIL), (cases.case_DT_small, S.KERNEL_CASH_TAIL),
                       (cases.case_TP_small, S.KERNEL_GENERIC), (cases.case_E_small, S.KERNEL_GENERIC)):
        spec, _ = case()
        assert S.Solver(spec).solve().stats()["kernel_used"] == used, spec.name


def test_cash_row_kernel_shapes(S, oracle):
    """bi_cash_row: several 128-level cash segments with a ragged last one, 0.1 and integer cash grids, K > 0 with a
    cash reserve, deposit and overhead rates, bankruptcy penalty, gamma < 1, survival recursion with per-period
    prices; whole grid against the oracle and the generic kernel."""
    specs = [
        S.cash_constraint_model(cases.pmf([4, 6, 5], 0.999), price=7, vari_cost=1.5, fixed_cost=3, hold_cost=0.25, salvage=0.5,
                                overhead=2, overhead_rate=0.05, deposit_rate=0.02, penalty_cost=0.3, max_order=11,
                                inv_min=0, inv_max=17, cash_min=0, cash_max=41.7, gamma=0.97),
        S.cash_constraint_model(cases.pmf([5, 5], 0.99), price=9, vari_cost=2, salvage=1, max_order=9, inv_min=0, inv_max=14,
                                cash_min=0, cash_max=300, quantiser=S.abi.Q_LONGDIV, q_mul=1.0, q_div=1.0, hold_cost=0.5),
        S.cash_survival_model(cases.pmf([5, 6, 4], 0.99), price_t=[4.5, 5, 4], vari_cost_t=[1, 1.5, 2], overhead_t=[11, 9, 12],
                              salvage=0.5, hold_cost=0.25, deposit_rate=0.01, max_order=12, inv_min=0, inv_max=20,
                              cash_min=-20, cash_max=150),
    ]
    # the overdraft lambdas (CashOverdraft.java:72-118) on an integer grid (long division by 10), on a 0.1 grid, with a
    # fixed cost / salvage / discount, and cash bounds that the clamp hits on both sides
    specs += [
        S.cash_overdraft_model(cases.pmf([6, 7, 5], 0.999), price=9, vari_cost=1, fixed_cost=4, salvage=1.5, overhead_t=[15, 18, 12],
                               r0=0.03, r2=0.11, r3=1.7, od_limit=25, interest_free=6, max_order=13, inv_min=0, inv_max=19,
                               cash_min=-45, cash_max=131, gamma=0.93),
        S.cash_overdraft_model(cases.pmf([5, 6], 0.99), price=8, vari_cost=2, overhead_t=[10, 10], r0=0.01, r2=0.125, r3=2.0,
                               od_limit=15, max_order=10, inv_min=0, inv_max=15, cash_min=-20.3, cash_max=37.9,
                               quantiser=S.abi.Q_DIV, q_mul=10.0, q_div=10.0),
    ]
    for n, spec in enumerate(specs):
        Vo, Qo, evals, _ = oracle.dense(spec)
        s, V, Q = _solve_all(S, spec)
        want = S.KERNEL_CASH_ROW if spec.recursion == S.REC_SURVIVAL else S.KERNEL_CASH_TAIL
        assert s.stats()["kernel_used"] == want and s.stats()["evals"] == evals, (n, spec.name)
        assert np.array_equal(V, Vo) and np.array_equal(Q, Qo), (n, spec.name)
        if want == S.KERNEL_CASH_TAIL:   # the older row kernel still agrees where it applies (as a request)
            r, Vr, Qr = _solve_all(S, spec, kernel=S.KERNEL_CASH_ROW)
            assert np.array_equal(Vr, Vo) and np.array_equal(Qr, Qo), (n, spec.name)
        g, Vg, Qg = _solve_all(S, spec, kernel=S.KERNEL_GENERIC)
        assert g.stats()["kernel_used"] == S.KERNEL_GENERIC
        assert np.array_equal(Vg, Vo) and np.array_equal(Qg, Qo), spec.name


@pytest.mark.parametrize("case", [cases.case_B1_ref, cases.case_B1_fixed, cases.case_B2_small],
                         ids=lambda f: f.__name__[5:])
@pytest.mark.parametrize("dedup", [False, True])
def test_staged_kernel_whole_grid(case, dedup, S, oracle):
    """bi_backorder_staged requested explicitly (AUTO prefers the slab kernel)."""
    spec, _ = case()
    Vo, Qo, _, _ = oracle.dense(spec)
    s, V, Q = _solve_all(S, spec, kernel=S.KERNEL_STAGED, dedup=dedup)
    assert np.array_equal(V, Vo) and np.array_equal(Q, Qo)
    assert s.stats()["kernel_used"] == S.KERNEL_STAGED


def test_lead_slab_wide_cases(S, oracle):
    """Slab-kernel tile edges: preQ counts that are not multiples of 8 / 4, D not a multiple of 4,
    lead time 1 and 2, clamped and unclamped, with and without folding."""
    for (lead, max_order, means, clamp) in [(2, 9, [3, 4, 3], True), (2, 12, [5, 2], True), (1, 21, [6, 7, 5], True),
                                            (1, 10, [3, 3, 3], False), (2, 4, [2, 2, 2], False)]:
        p = S.poisson_pmf(means, 0.999)
        dmax = max(r[-1, 0] for r in p)
        T = len(means)
        inv_min, inv_max = (-T * dmax, T * max_order) if not clamp else (-14, 17)
        spec = S.leadtime_model(p, fixed_cost=4, vari_cost=1, hold_cost=2, penalty_cost=9, max_order=max_order,
                                inv_min=inv_min, inv_max=inv_max, lead_time=lead, clamp=clamp)
        Vo, Qo, _, _ = oracle.dense(spec)
        for dedup in (False, True):
            auto = S.KERNEL_LEAD_Q2 if lead == 2 and not dedup else S.KERNEL_LEAD_COL
            for k, used in ((S.KERNEL_AUTO, auto), (S.KERNEL_LEAD_COL, S.KERNEL_LEAD_COL),
                            (S.KERNEL_LEAD_SLAB, S.KERNEL_LEAD_SLAB)):
                s, V, Q = _solve_all(S, spec, dedup=dedup, kernel=k)
                assert s.stats()["kernel_used"] == used
                assert np.array_equal(V, Vo) and np.array_equal(Q, Qo), (lead, max_order, clamp, dedup, k)


def test_staged_kernel_is_used_for_leadtime(S):
    spec, _ = cases.case_B2_small()
    assert S.Solver(spec).solve().stats()["kernel_used"] == S.KERNEL_LEAD_Q2
    assert S.Solver(spec, kernel=S.KERNEL_LEAD_COL).solve().stats()["kernel_used"] == S.KERNEL_LEAD_COL
    assert S.Solver(spec, kernel=S.KERNEL_LEAD_SLAB).solve().stats()["kernel_used"] == S.KERNEL_LEAD_SLAB
    with pytest.raises(S.SdpbError):  # folded grids and lead time 1 have no all-actions-in-thread kernel
        S.Solver(spec, kernel=S.KERNEL_LEAD_Q2, dedup=True)
    with pytest.raises(S.SdpbError):
        S.Solver(cases.case_B1_ref()[0], kernel=S.KERNEL_LEAD_Q2)
    assert S.Solver(spec, kernel=S.KERNEL_STAGED).solve().stats()["kernel_used"] == S.KERNEL_STAGED
    assert S.Solver(spec, kernel=S.KERNEL_GENERIC).solve().stats()["kernel_used"] == S.KERNEL_GENERIC
    spec, _ = cases.case_A_small()
    assert S.Solver(spec).solve().stats()["kernel_used"] == S.KERNEL_FUSED  # small grid: the whole horizon in one launch
    assert S.Solver(spec, kernel=S.KERNEL_TILED).solve().stats()["kernel_used"] == S.KERNEL_TILED


@pytest.mark.parametrize("case", A_CASES, ids=lambda f: f.__name__[5:])
def test_fused_whole_horizon_kernel(case, S, oracle):
    """bi_inv_fused: one cooperative launch for all periods (small unsharded 1-D grids).  Whole grid against the
    oracle, repeated solves, and the per-period API (which keeps using the per-period kernels) on the same handle."""
    spec, init = case()
    Vo, Qo, evals, _ = oracle.dense(spec)
    if spec.flags & S.abi.F_GY_MODE:
        with pytest.raises(S.SdpbError):
            S.Solver(spec, kernel=S.KERNEL_FUSED)
        return
    s, V, Q = _solve_all(S, spec, kernel=S.KERNEL_FUSED)
    st = s.stats()
    assert st["kernel_used"] == S.KERNEL_FUSED and st["launches"] == 1 and st["evals"] == evals
    assert np.array_equal(V, Vo) and np.array_equal(Q, Qo)
    for _ in range(2):
        s.solve()
        V1, Q1 = s.period_tables(1)
        assert np.array_equal(V1, Vo[0]) and np.array_equal(Q1, Qo[0])
    for t in range(spec.T, 0, -1):
        s.solve_period_async(t)
    s.sync()
    V1, Q1 = s.period_tables(1)
    assert np.array_equal(V1, Vo[0]) and np.array_equal(Q1, Qo[0])


def test_fused_kernel_shapes(S, oracle):
    """States not a multiple of the CTA slice, more states than SMs (several states per CTA), fewer states than
    SMs, MAX direction, sparse demand support, action counts around the 8-pair batch and the 32-lane argopt."""
    rng = np.random.default_rng(3)
    for n_states, n_act, direction in ((149, 33, S.abi.MIN), (700, 9, S.abi.MAX), (2001, 40, S.abi.MIN), (37, 257, S.abi.MIN),
                                       (5000, 3, S.abi.MIN)):
        rows = []
        for _ in range(3):
            sup = np.sort(rng.choice(np.arange(0, 14), size=int(rng.integers(2, 9)), replace=False)).astype(float)
            rows.append(np.column_stack([sup, rng.dirichlet(np.ones(len(sup)))]))
        half = n_states // 2
        spec = S.inventory_model(rows, fixed_cost=7, vari_cost=1, hold_cost=1, penalty_cost=6, max_order=n_act - 1,
                                 inv_min=-half, inv_max=n_states - half - 1, direction=direction)
        Vo, Qo, evals, _ = oracle.dense(spec)
        s, V, Q = _solve_all(S, spec, kernel=S.KERNEL_FUSED)
        assert s.stats()["kernel_used"] == S.KERNEL_FUSED
        assert np.array_equal(V, Vo) and np.array_equal(Q, Qo), (n_states, n_act)
    with pytest.raises(S.SdpbError):
        S.Solver(cases.case_B1_ref()[0], kernel=S.KERNEL_FUSED)
    # AUTO: C1 (1,001 states) runs fused, C2 (2,001 x 101) stays on the per-period tiled kernel; same tables either way
    assert S.Solver(S.configs.c1()).solve().stats()["kernel_used"] == S.KERNEL_FUSED
    spec = S.configs.c2()
    a, Va, Qa = _solve_all(S, spec)
    f, Vf, Qf = _solve_all(S, spec, kernel=S.KERNEL_FUSED)
    assert a.stats()["kernel_used"] == S.KERNEL_TILED and f.stats()["kernel_used"] == S.KERNEL_FUSED
    assert np.array_equal(Va, Vf) and np.array_equal(Qa, Qf)


@pytest.mark.parametrize("name", cases.GOLDEN)
def test_against_golden_fixtures(name, S):
    spec, init, g = cases.load_golden(name)
    s, V, Q = _solve_all(S, spec)
    per = g["periods"] - 1
    assert np.array_equal(V[per], g["V"])
    assert np.array_equal(Q[per].astype(np.float32), g["Q"])
    v, q = s.value(1, g["init"])
    assert np.array_equal(v, g["init_values"])


@pytest.mark.parametrize("case", cases.ALL, ids=lambda f: f.__name__[5:])
def test_value_and_opt_table_match_topdown(case, S, oracle):
    """getExpectedValue/getAction and the getOptTable() row set (visited states only, sorted)."""
    spec, init = case()
    rows, iv, _ = oracle.topdown(spec, init)
    s = S.Solver(spec).solve()
    v, q = s.value(1, init)
    assert np.array_equal(v, iv)
    s.reach(init)
    tab = s.opt_table()
    nd = spec.ndim
    assert tab.shape == (len(rows), nd + 2)
    # the oracle emits rows in the memo-map order (period, inv, preQ.., cash); the library in its
    # grid order, which is the same ordering
    assert np.array_equal(tab[:, :nd + 1], rows[:, :nd + 1])
    assert np.array_equal(tab[:, -1], rows[:, -2])
    # every visited state answers through sdpb_value too
    for t in range(1, spec.T + 1):
        sel = rows[rows[:, 0] == t]
        if len(sel):
            v, q = s.value(t, sel[:, 1:1 + nd])
            assert np.array_equal(v, sel[:, -1]) and np.array_equal(q, sel[:, -2])


@pytest.mark.parametrize("case", cases.ALL, ids=lambda f: f.__name__[5:])
def test_device_lambdas_match_oracle(case, S, oracle):
    """sdpb_eval_triples (the device code of c, f, |A|) against the oracle's lambdas."""
    import random
    spec, _ = case()
    if spec.two_product or spec.staff:
        pytest.skip("sdpb_eval_triples is not implemented for the two-product and staff kinds")
    pkg = S.package
    from importlib import import_module
    spot = import_module(pkg.__name__ + "._spot")
    rng = random.Random(7)
    s = S.Solver(spec)
    for _ in range(60):
        st, a, d = spot.random_triple(spec, rng)
        c, nxt, na = spot.eval_descriptor(spec, st, a, d, solver=s)
        assert na == oracle.n_actions(spec, st[0], st[1:])
        co, no = oracle.eval_triple(spec, st[0], st[1:], a, d)
        assert c == co
        if st[0] < spec.T and oracle.index(spec, no) >= 0:
            assert tuple(no) == nxt


def test_repeated_solves_replay_a_cuda_graph(S, oracle):
    """From the second sdpb_solve on, the T launches are one captured graph: results must not change."""
    for case in (cases.case_A_small, cases.case_C_int, cases.case_B2_small):
        spec, init = case()
        Vo, Qo, evals, _ = oracle.dense(spec)
        s = S.Solver(spec)
        for rep in range(4):
            s.solve()
            for t in (1, spec.T):
                V, Q = s.period_tables(t)
                assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), (spec.name, rep, t)
            assert s.stats()["evals"] == evals
        s.solve_async()
        s.sync()
        v, _ = s.value(1, init)
        assert v[0] == Vo[0][oracle.index(spec, init[0])]


@pytest.mark.parametrize("case", [cases.case_A_small, cases.case_B1_fixed, cases.case_B2_small, cases.case_C_rich,
                                  cases.case_C_int, cases.case_D_rich, cases.case_E_small, cases.case_XR_small,
                                  cases.case_DT_small, cases.case_TP_small], ids=lambda f: f.__name__[5:])
def test_policy_rollout_matches_oracle(case, S, oracle):
    """sdpb_simulate (Simulation.java:59-70) against the oracle's roll-out of its own policy tables,
    path by path, on seeded samples that include out-of-support demands and non-integer draws."""
    spec, init = case()
    Vo, Qo, _, _ = oracle.dense(spec)
    rng = np.random.default_rng(5)
    dmax = max(r[-1, 0] for r in spec.pmf)
    samples = rng.uniform(-0.4, dmax + 3.0, size=(500, spec.T))
    gamma = spec.gamma
    s = S.Solver(spec).solve()
    got = s.simulate(init[0], samples, gamma)
    want = oracle.simulate(spec, Qo, init[0], samples, gamma)
    assert np.array_equal(got, want)


def test_reference_style_simulation(S, oracle):
    """Reads like CLSPTesting.java:125-127: Simulation(distributions, sampleNum, recursion)."""
    dists = [S.PoissonDist(m) for m in (5, 8, 6)]
    pmf = S.GetPmf(dists, 0.999, 1).getpmf()
    spec = S.inventory_model(pmf, 20, 1, 1, 5, max_order=15, inv_min=-30, inv_max=30)
    recursion = S.Recursion(spec)
    sim = S.Simulation(dists, 2000, recursion)
    samples = S.generate_lh_samples(dists, 2000)
    mean = sim.simulateSDPGivenSamplNum(S.State(1, 0), samples)
    opt = recursion.getExpectedValue(S.State(1, 0))
    assert abs(mean - opt) / opt < 0.05          # the reference's eyeball check: simulated ~ optimal
    Vo, Qo, _, _ = oracle.dense(spec)
    assert np.array_equal(sim.simulate_paths(S.State(1, 0), samples), oracle.simulate(spec, Qo, [0.0], samples))


GROUP_CASES = [(cases.case_A_small, 2), (cases.case_A_gy, 3), (cases.case_B2_small, 3), (cases.case_B1_ref, 2),
               (cases.case_B1_fixed, 4), (cases.case_C_int, 3), (cases.case_C_rich, 2), (cases.case_C_small, 5),
               (cases.case_D_small, 3), (cases.case_F_small, 2), (cases.case_E_small, 2), (cases.case_M2_small, 3),
               (cases.case_W_small, 2), (cases.case_XR_small, 2), (cases.case_A_terminal, 3), (cases.case_B2_terminal, 4),
               (cases.case_C_terminal, 3), (cases.case_M2_terminal, 2), (cases.case_A_one_state, 3),
               (cases.case_C_int_tall, 2), (cases.case_C_int_tall, 3)]


@pytest.mark.parametrize("case,world", GROUP_CASES, ids=lambda x: getattr(x, "__name__", str(x))[5:])
def test_group_on_one_gpu(case, world, S, oracle):
    """The multi-GPU data path inside the library, on one device: sdpb_group_create cuts the grid into `world` shards
    (here all on GPU 0), each holding only its window of V_t; after every period the shards copy the rows their peers
    read straight into the peers' tables and hand over with device-side flags.  Whole grid, every period, against the
    oracle; per-shard windows, traffic and evaluation counts."""
    spec, init = case()
    Vo, Qo, evals, _ = oracle.dense(spec)
    n = Vo.shape[1]
    with S.Group(spec, [0] * world) as g:
        g.solve()
        g.solve()  # a second solve on the same tables: the flag epochs keep counting
        for t in range(1, spec.T + 1):
            V, Q = g.period_tables(t)
            assert np.array_equal(V, Vo[t - 1]), t
            assert np.array_equal(Q, Qo[t - 1]), t
        assert g.stats()["evals"] == evals
        v, q = g.value(1, init)
        rows, iv, _ = oracle.topdown(spec, init)
        assert np.array_equal(v, iv)
        par = S.package.parallel
        for r, sh in enumerate(g.shards):
            lo, hi, _ = par.shard_bounds(n, r, world)
            gi = sh.grid
            assert (gi.shard_lo, gi.shard_hi) == (lo, hi)
            need = sh.shard_reads()
            assert need == par.needed_range(spec, lo, hi, n)
            if hi > lo:
                assert gi.window_lo <= min(need[0], lo) and gi.window_hi >= max(need[1], hi)
                Vb, Qb = sh.shard_tables(1)
                assert np.array_equal(Vb, Vo[0][lo:hi]) and np.array_equal(Qb, Qo[0][lo:hi])


def test_group_kernel_choices_on_one_gpu(S, oracle):
    """Every specialised kernel under sharding: block edges that cut through tiles, rows and diagonals."""
    jobs = [(cases.case_B2_small, 3, S.KERNEL_GENERIC), (cases.case_B2_small, 5, S.KERNEL_STAGED),
            (cases.case_B2_small, 3, S.KERNEL_LEAD_SLAB), (cases.case_B2_small, 4, S.KERNEL_LEAD_COL),
            (cases.case_B2_small, 7, S.KERNEL_LEAD_Q2), (cases.case_C_int, 4, S.KERNEL_CASH_INT),
            (cases.case_C_int_K, 5, S.KERNEL_AUTO), (cases.case_A_small, 4, S.KERNEL_TILED),
            (cases.case_A_small, 3, S.KERNEL_TILED2), (cases.case_A_terminal_big, 3, S.KERNEL_TILED2),
            (cases.case_A_terminal_big, 7, S.KERNEL_TILED)]
    for case, world, kernel in jobs:
        spec, _ = case()
        Vo, Qo, _, _ = oracle.dense(spec)
        with S.Group(spec, [0] * world, kernel=kernel) as g:
            g.solve()
            for t in range(1, spec.T + 1):
                V, Q = g.period_tables(t)
                assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), (spec.name, world, kernel, t)


def test_group_dedup_on_one_gpu(S, oracle):
    spec, _ = cases.case_B2_small()
    Vo, Qo, _, _ = oracle.dense(spec)
    with S.Group(spec, [0, 0, 0], dedup=True) as g:
        g.solve()
        for t in range(1, spec.T + 1):
            V, Q = g.period_tables(t)
            assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1])


def test_large_group_c5_on_one_gpu(S, oracle):
    """tiled2 with shard boundaries that cut through 1021-state tiles; each shard holds about a third of the memory."""
    spec = S.configs.c5(n_states=300_007, T=3, n_actions=37)
    ref = S.Solver(spec).solve()
    full_bytes = ref.grid.device_bytes
    with S.Group(spec, [0, 0, 0], kernel=S.KERNEL_TILED2, profile=True) as g:
        g.solve()
        assert g.shards[0].stats()["kernel_used"] == S.KERNEL_TILED2
        for t in (1, 2, 3):
            Vr, Qr = ref.period_tables(t)
            V, Q = g.period_tables(t)
            assert np.array_equal(V, Vr) and np.array_equal(Q, Qr)
        for sh in g.shards:
            assert sh.grid.device_bytes < 0.40 * full_bytes        # the window, not the whole table
            out_b, in_b = sh.peer_traffic()
            assert 0 < out_b < 64 * 1024 and 0 < in_b < 64 * 1024  # a halo of a few hundred states
            prof = sh.period_profile()
            assert prof.shape == (3, 3) and (prof[:, 0] > 0).all()


def _ipc_worker(rank, world, case_name, kernel, q_in, q_out, out_dir, same_gpu=False):
    """One process per shard, shard r on GPU r: the torchrun layout, connected through CUDA IPC."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import numpy as np
    import cases as cs
    import sdpb200 as S_
    spec, _ = getattr(cs, case_name)()
    s = S_.Solver(spec, device=0 if same_gpu else rank, shard_rank=rank, shard_count=world, kernel=kernel)
    q_out.put((rank, s.peer_export()))
    blobs = q_in.get()
    if same_gpu:
        try:
            s.peer_attach(blobs)
            q_out.put((rank, b"attached"))
        except S_.SdpbError as e:
            q_out.put((rank, b"refused" if e.code == S_.abi.SDPB_ERR_PEER else b"other"))
        q_in.get()
        s.close()
        return
    s.peer_attach(blobs)
    for _ in range(2):
        s.solve()
    res = {}
    for t in range(1, spec.T + 1):
        V, Q = s.shard_tables(t)
        res[f"V{t}"], res[f"Q{t}"] = V, Q
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), lo=s.grid.shard_lo, hi=s.grid.shard_hi, **res)
    q_out.put((rank, b"done"))
    q_in.get()  # keep the tables alive until every shard has finished
    s.close()


@pytest.mark.parametrize("case_name,world,kernel", [("case_B2_small", 3, 0), ("case_C_int", 2, 0), ("case_A_small", 2, 0)])
def test_ipc_shards_in_separate_processes(case_name, world, kernel, S, oracle, tmp_path):
    """sdpb_peer_export / sdpb_peer_attach across PROCESSES (cudaIpcOpenMemHandle), the layout bench.py runs under
    torchrun: one process per GPU.  Needs as many GPUs as shards (processes that spin on each other's flags must not
    share a GPU); on a one-GPU box the same path is exercised by bench.py --gpus N (verified_vs_unsharded)."""
    import multiprocessing as mp
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    ctx = mp.get_context("spawn")
    q_out = ctx.Queue()
    q_ins = [ctx.Queue() for _ in range(world)]
    procs = [ctx.Process(target=_ipc_worker, args=(r, world, case_name, kernel, q_ins[r], q_out, str(tmp_path)))
             for r in range(world)]
    for p in procs:
        p.start()
    try:
        blobs = dict(q_out.get(timeout=180) for _ in range(world))
        for qi in q_ins:
            qi.put([blobs[r] for r in range(world)])
        for _ in range(world):
            assert q_out.get(timeout=180)[1] == b"done"
        for qi in q_ins:
            qi.put("bye")
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
    spec, _ = getattr(cases, case_name)()
    Vo, Qo, _, _ = oracle.dense(spec)
    covered = 0
    for r in range(world):
        gz = np.load(tmp_path / f"r{r}.npz")
        lo, hi = int(gz["lo"]), int(gz["hi"])
        for t in range(1, spec.T + 1):
            assert np.array_equal(gz[f"V{t}"], Vo[t - 1][lo:hi]), (r, t)
            assert np.array_equal(gz[f"Q{t}"], Qo[t - 1][lo:hi]), (r, t)
        covered += hi - lo
    assert covered == Vo.shape[1]


# ---- dense-grid artefacts at visited states: reported, not silent -----------------------------------------------
def _unclamped_leadtime(S, inv_min, inv_max, T=3, mean=4, maxq=12):
    return S.leadtime_model(cases.pmf([mean] * T), fixed_cost=0, vari_cost=1, hold_cost=2, penalty_cost=10,
                            max_order=maxq, inv_min=inv_min, inv_max=inv_max, lead_time=1, clamp=False)


def test_reach_reports_clipped_successors(S, oracle):
    """Leadtime.java:63-67 does not clamp: on a grid smaller than the reachable hull the kernels fold successors onto
    the boundary row.  sdpb_reach says so (SDPB_ERR_OFFGRID) when a state the reference visits is affected, unless the
    caller allows it; with the hull from sdpb_reachable_hull nothing is clipped and the values are the reference's."""
    init = [[0.0, 0.0]]
    small = _unclamped_leadtime(S, -8, 20)
    s = S.Solver(small).solve()
    with pytest.raises(S.SdpbError) as e:
        s.reach(init)
    assert e.value.code == S.abi.SDPB_ERR_OFFGRID and "outside the inventory grid" in str(e.value)
    assert s.stats()["clipped_successors"] > 0
    with pytest.raises(S.SdpbError):                       # the facade refuses too
        S.LeadtimeRecursion(small).getExpectedValue(S.LeadtimeState(1, 0.0, 0.0))
    ok = S.Solver(small, allow=S.ALLOW_CLIPPED_SUCCESSORS).solve()
    ok.reach(init)                                         # opt-out: counted, not refused
    assert ok.stats()["clipped_successors"] == s.stats()["clipped_successors"]
    # the dense oracle counts the same event over the WHOLE grid, so it sees at least as many
    assert oracle.dense(small)[3] >= ok.stats()["clipped_successors"]

    lo, hi = S.reachable_hull(small, init)
    assert lo == -2 * max(r[-1, 0] for r in small.pmf) and hi == 24.0
    hull = _unclamped_leadtime(S, lo, hi)
    rec = S.LeadtimeRecursion(hull)
    v = rec.getExpectedValue(S.LeadtimeState(1, 0.0, 0.0))   # runs sdpb_reach: passes
    assert rec.stats()["clipped_successors"] == 0
    rows, iv, _ = oracle.topdown(hull, init)               # the reference's control flow: unbounded real-valued states
    assert v == iv[0]
    tab = rec.getOptTable()
    assert np.array_equal(tab, rows[:, :-1])
    # a clamped model never reports anything
    c = S.Solver(cases.case_B1_fixed()[0]).solve()
    c.reach([[0.0, 0.0]])
    assert c.stats()["clipped_successors"] == 0


def test_reach_reports_capped_action_sets(S, oracle):
    capped, init = cases.case_XR_small()
    capped.allow = 0
    s = S.Solver(capped).solve()
    with pytest.raises(S.SdpbError) as e:
        s.reach(init)
    assert e.value.code == S.abi.SDPB_ERR_OFFGRID and "order-up-to" in str(e.value)
    assert s.stats()["capped_action_sets"] > 0
    spec, init = cases.case_XR_uncapped()
    u = S.Solver(spec).solve()
    u.reach(init)
    assert u.stats()["capped_action_sets"] == 0


def test_strict_cash_bounds(S):
    spec, init = cases.case_C_int()
    s = S.Solver(spec, strict_cash_bounds=True).solve()
    with pytest.raises(S.SdpbError) as e:                  # cash_max = 260 is reached from (0, 12) within 4 periods
        s.reach(init)
    assert e.value.code == S.abi.SDPB_ERR_OFFGRID and s.stats()["cash_bound_hits"] > 0
    lax = S.Solver(spec).solve()
    lax.reach(init)                                        # the clamp is part of the reference lambdas: fine by default
    assert lax.stats()["cash_bound_hits"] == s.stats()["cash_bound_hits"]


@pytest.mark.parametrize("case", cases.NOLAST, ids=lambda f: f.__name__[5:])
def test_no_order_last_auto_equals_generic(case, S, oracle):
    """SDPB_F_NO_ORDER_LAST on the families whose fast kernels do not know the rule: period T must take the general
    path, every other period the specialised one; AUTO == GENERIC == oracle, counts included."""
    spec, init = case()
    Vo, Qo, evals, _ = oracle.dense(spec)
    assert np.all(Qo[-1] == 0)
    a, Va, Qa = _solve_all(S, spec)
    g, Vg, Qg = _solve_all(S, spec, kernel=S.KERNEL_GENERIC)
    assert np.array_equal(Va, Vo) and np.array_equal(Qa, Qo)
    assert np.array_equal(Vg, Vo) and np.array_equal(Qg, Qo)
    assert a.stats()["evals"] == g.stats()["evals"] == evals
    assert a.stats()["kernel_used"] != S.KERNEL_GENERIC   # the other periods still ran on the fast kernel
    if spec.lead_time:
        d, Vd, Qd = _solve_all(S, spec, dedup=True)
        assert np.array_equal(Vd, Vo) and np.array_equal(Qd, Qo)


def test_boundary_function_facade(S, oracle):
    """Reads like MultiItemCashXW.java:118-121 / CashRecursionV.java:125-128 for one product: the engine takes a
    BoundaryFuncton lambda and values the states of period T+1 with it."""
    spec = S.cash_constraint_model(cases.pmf([5, 6, 5]), price=10, vari_cost=1, salvage=0.0, max_order=14, inv_min=0,
                                   inv_max=25, cash_min=0, cash_max=200, quantiser=S.Q_LONGDIV, q_mul=1.0, q_div=1.0)
    salPrice = 0.5
    boundFinalCash = lambda iniInventory, iniCash: iniCash + salPrice * iniInventory  # noqa: E731
    recursion = S.CashRecursion(spec, boundFinalCash=boundFinalCash)
    ref, init = cases.case_C_terminal()
    rows, iv, _ = oracle.topdown(ref, init)
    iniState = S.CashState(1, init[0][0], init[0][1])
    assert recursion.getExpectedValue(iniState) == iv[0]
    assert recursion.getAction(iniState) == rows[0][-2]
    # without the boundary function the answer is a different one
    assert S.CashRecursion(spec).getExpectedValue(iniState) != iv[0]


def test_multi_gpu_facade_on_one_gpu(S, oracle):
    spec, init = cases.case_B2_small()
    rows, iv, _ = oracle.topdown(spec, init)
    rec = S.LeadtimeRecursion2(spec, devices=[0, 0, 0])
    st = S.LeadtimeRecursion2.state_cls(1, 0.0, 0.0, 0.0)
    assert rec.getExpectedValue(st) == iv[0] and rec.getAction(st) == rows[0][-2]


def test_solve_batch(S, oracle):
    """sdpb_solve_batch: many small independent instances (the parameter sweeps of CLSPTesting.java:57-61) solved
    together; first call plain, second call captures one CUDA graph for the whole batch, third call replays it."""
    specs = []
    for k in range(12):
        specs.append(S.inventory_model(cases.pmf([5 + k % 3, 8, 6 + k % 2]), fixed_cost=20 + 5 * k, vari_cost=1,
                                       hold_cost=1 + 0.5 * (k % 2), penalty_cost=5 + k, max_order=15 + k,
                                       inv_min=-30 - k, inv_max=30 + 2 * k))
    specs.append(cases.case_B2_small()[0])      # any unsharded handle may be in a batch
    specs.append(cases.case_C_int()[0])
    solvers = [S.Solver(sp, kernel=S.KERNEL_TILED if sp.cost_kind == S.COST_BACKORDER and sp.lead_time == 0 else S.KERNEL_AUTO)
               for sp in specs]
    for rep in range(4):
        S.solve_batch(solvers)
        if rep in (0, 2, 3):
            for sp, s in zip(specs, solvers):
                Vo, Qo, evals, _ = oracle.dense(sp)
                for t in range(1, sp.T + 1):
                    V, Q = s.period_tables(t)
                    assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), (rep, sp.name, t)
                assert s.stats()["evals"] == evals
    # AUTO handles (the fused whole-horizon kernel on these sizes) batch too
    auto = [S.Solver(sp) for sp in specs[:6]]
    for _ in range(3):
        S.solve_batch(auto)
    for sp, s in zip(specs[:6], auto):
        Vo, Qo, _, _ = oracle.dense(sp)
        V, Q = s.period_tables(1)
        assert np.array_equal(V, Vo[0]) and np.array_equal(Q, Qo[0])


def test_solve_batch_wide(S, oracle):
    """A batch wide enough to fill the GPU by itself (72 instances): the library then runs every instance on the 2-D
    register tile with a small action split; three rounds (plain, capture, replay)."""
    specs = [S.inventory_model(cases.pmf([5 + k % 3, 8 + k % 4, 6 + k % 2]), fixed_cost=20 + 5 * (k % 6), vari_cost=k % 2,
                               hold_cost=1 + 0.5 * (k % 2), penalty_cost=5 + k % 5, max_order=15 + k % 7,
                               inv_min=-30 - k % 5, inv_max=30 + 2 * (k % 9)) for k in range(8)]
    want = [oracle.dense(sp) for sp in specs]
    solvers = [S.Solver(specs[k % 8]) for k in range(72)]
    for rep in range(3):
        S.solve_batch(solvers)
    for k, s in enumerate(solvers):
        Vo, Qo, evals, _ = want[k % 8]
        for t in range(1, specs[k % 8].T + 1):
            V, Q = s.period_tables(t)
            assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), (k, t)
        assert s.stats()["evals"] == evals
    assert solvers[0].stats()["kernel_used"] in (S.KERNEL_TILED2, S.KERNEL_FUSED, S.KERNEL_TILED)
    for s in solvers:
        s.close()


@pytest.mark.parametrize("mode", ["default", "share", "split2", "split4"])
def test_lead_q2m_forced(mode):
    """The lead-time-2 kernels on 16 small random instances, unsharded and as a three-shard group: as the library shapes
    the launch by itself (bi_lead_q2m with action slices over separate CTAs + merge kernel), and forced by one test hook
    each to bi_lead_q2m without action slices (share) and to bi_lead_q2 with 2 or 4 thread groups (split2, split4).
    The hooks are read once per process, hence the subprocess."""
    import os
    import subprocess
    import sys
    env = dict(os.environ)
    env.pop("SDPB_Q2_SHARE", None), env.pop("SDPB_Q2_SPLIT", None)
    # default: on these small grids the library cuts the action range over separate CTAs (gridDim.y) and merges with
    # merge_action_slices -- the path the multi-GPU shards of C4 take
    if mode == "share":
        env["SDPB_Q2_SHARE"] = "1"
    elif mode.startswith("split"):
        env["SDPB_Q2_SPLIT"] = mode[len("split"):]
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "q2m_worker.py")
    r = subprocess.run([sys.executable, worker], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "16 instances ok" in r.stdout


def test_collapsed_kernel_is_opt_in_and_close(S, oracle):
    """SDPB_KERNEL_COLLAPSED: G(y) per order-up-to level, then V(x) = opt_a cost(a) + G(x + a).  Opt-in, NOT bit-identical:
    values within 1e-9 relative of the oracle (observed ~1e-13), the policy equal except between near-tied actions;
    never chosen by AUTO; refused for models it does not cover."""
    for case in (cases.case_A_small, cases.case_A_max, cases.case_A_twopoint, cases.case_A_halfstep,
                 cases.case_A_sparse_pmf, cases.case_A_degenerate, cases.case_A_one_state, cases.case_A_terminal,
                 cases.case_CLSP_main):
        spec, _ = case()
        Vo, Qo, evals, _ = oracle.dense(spec)
        with S.Solver(spec, kernel=S.KERNEL_COLLAPSED) as s:
            s.solve()
            s.solve()   # the second solve replays the captured graph
            st = s.stats()
            assert st["kernel_used"] == S.KERNEL_COLLAPSED and st["evals"] == evals
            agree = total = 0
            for t in range(1, spec.T + 1):
                V, Q = s.period_tables(t)
                np.testing.assert_allclose(V, Vo[t - 1], rtol=1e-9, atol=1e-9, err_msg=f"{spec.name} t={t}")
                agree += int((Q == Qo[t - 1]).sum())
                total += Q.size
            assert agree >= 0.98 * total, (spec.name, agree, total)
        with S.Solver(spec) as s:                           # AUTO never picks it
            assert s.solve().stats()["kernel_used"] != S.KERNEL_COLLAPSED
    # a large grid against the exact GPU solve: C5 at 1e6 states
    spec = S.configs.c5(n_states=1_000_000, T=3)
    with S.Solver(spec) as ex, S.Solver(spec, kernel=S.KERNEL_COLLAPSED) as co:
        ex.solve(), co.solve()
        for t in range(1, spec.T + 1):
            Ve, Qe = ex.period_tables(t)
            Vc, Qc = co.period_tables(t)
            np.testing.assert_allclose(Vc, Ve, rtol=1e-9)
            assert (Qc == Qe).mean() > 0.999
        assert co.stats()["evals"] == ex.stats()["evals"] and co.stats()["evals_executed"] < 0.02 * ex.stats()["evals"]
    # refused where it does not apply
    for bad in (cases.case_B2_small()[0], cases.case_C_int()[0], cases.case_A_nolast()[0], cases.case_A_gy()[0]):
        with pytest.raises(S.SdpbError) as e:
            S.Solver(bad, kernel=S.KERNEL_COLLAPSED)
        assert e.value.code == S.abi.SDPB_ERR_ARG
    with pytest.raises(S.SdpbError):
        S.Solver(cases.case_A_small()[0], kernel=S.KERNEL_COLLAPSED, shard_rank=0, shard_count=2)


def test_reference_style_driver_clsp_main(S, oracle):
    """Reads like src/capacitated/CLSP.java:196-290 (the self-contained demo with its own inline pmf)."""
    meanDemand = [9, 23, 53, 29]
    truncationQuantile, stepSize, minState, maxState = 0.99999, 1, -300, 300
    fixedOrderingCost, proportionalOrderingCost, holdingCost, penaltyCost, maxOrderQuantity = 500, 0, 2, 10, 60
    pmf = S.clsp_inline_pmf(meanDemand, truncationQuantile, stepSize)
    assert pmf[2][0, 0] > 0                                  # no LB = 0 override: Poisson(53) starts well above zero
    spec = S.inventory_model(pmf, fixedOrderingCost, proportionalOrderingCost, holdingCost, penaltyCost,
                             max_order=maxOrderQuantity, inv_min=minState, inv_max=maxState)
    inventory = S.Recursion(spec)
    initialState = S.State(1, 1)
    finalValue = inventory.getExpectedValue(initialState)
    rows, iv, _ = oracle.topdown(spec, [[1.0]])
    assert finalValue == iv[0] and inventory.getAction(initialState) == rows[0][-2]
    assert np.array_equal(inventory.getOptTable(), rows[:, :-1])


def test_processes_sharing_a_gpu_are_refused(S, tmp_path):
    """Two PROCESSES on one GPU would have to spin on each other's flags from kernels that are not guaranteed to run
    at the same time: sdpb_peer_attach refuses (SDPB_ERR_PEER) before anything is launched."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    q_out = ctx.Queue()
    q_ins = [ctx.Queue() for _ in range(2)]
    procs = [ctx.Process(target=_ipc_worker, args=(r, 2, "case_A_small", 0, q_ins[r], q_out, str(tmp_path), True))
             for r in range(2)]
    for p in procs:
        p.start()
    try:
        blobs = dict(q_out.get(timeout=180) for _ in range(2))
        for qi in q_ins:
            qi.put([blobs[r] for r in range(2)])
        answers = [q_out.get(timeout=180)[1] for _ in range(2)]
        for qi in q_ins:
            qi.put("bye")
        for p in procs:
            p.join(timeout=60)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
    assert answers == [b"refused", b"refused"]


def test_unattached_shard_refuses_to_solve(S):
    spec, _ = cases.case_A_small()
    s = S.Solver(spec, shard_rank=0, shard_count=2)
    with pytest.raises(S.SdpbError) as e:
        s.solve()
    assert e.value.code == S.abi.SDPB_ERR_STATE



def test_unsolved_state_raises(S):
    spec, _ = cases.case_A_small()
    s = S.Solver(spec)
    with pytest.raises(S.SdpbError) as e:
        s.value(1, [[0.0]])
    assert e.value.code == S.abi.SDPB_ERR_STATE
    s.solve()
    with pytest.raises(S.SdpbError) as e:
        s.value(1, [[1000.0]])  # outside the grid: Java would throw from getAction
    assert e.value.code == S.abi.SDPB_ERR_UNSOLVED
    with pytest.raises(S.SdpbError):
        s.value(1, [[0.25]])    # not a grid point


def test_reference_style_driver_capacitated(S, oracle):
    """Reads like src/capacitated/CLSPTesting.java:75-120: build pmf, lambdas, Recursion, solve."""
    pmf = S.GetPmf([S.PoissonDist(m) for m in (5, 8, 6)], 0.999, 1).getpmf()
    K, v, h, pi, maxQ, lo, hi = 20.0, 1.0, 1.0, 5.0, 15, -30.0, 30.0

    def getFeasibleAction(s):
        return [float(i) for i in range(maxQ + 1)]

    def stateTransition(state, action, randomDemand):
        nxt = state.getIniInventory() + action - randomDemand
        nxt = hi if nxt > hi else nxt
        nxt = lo if nxt < lo else nxt
        return S.State(state.getPeriod() + 1, nxt)

    def immediateValue(state, action, randomDemand):
        fixed = K if action > 0 else 0
        lvl = state.getIniInventory() + action - randomDemand
        return fixed + v * action + h * max(lvl, 0) + pi * max(-lvl, 0)

    spec = S.inventory_model(pmf, K, v, h, pi, max_order=maxQ, inv_min=lo, inv_max=hi)
    recursion = S.Recursion(spec, getFeasibleAction, stateTransition, immediateValue)
    with pytest.raises(KeyError):
        recursion.getAction(S.State(1, 0))      # NullPointerException in the reference
    initialState = S.State(1, 0)
    finalValue = recursion.getExpectedValue(initialState)
    rows, iv, _ = oracle.topdown(spec, [[0.0]])
    assert finalValue == iv[0]
    assert recursion.getAction(initialState) == rows[0][-2]
    assert np.array_equal(recursion.getOptTable(), rows[:, :3])
    acts = recursion.getCacheActions()
    assert len(acts) == len(rows) and acts[S.State(1, 0)] == rows[0][-2]
    # a wrong descriptor is caught by the spot check
    wrong = S.inventory_model(pmf, K, v, h, pi + 1, max_order=maxQ, inv_min=lo, inv_max=hi)
    with pytest.raises(ValueError):
        S.Recursion(wrong, getFeasibleAction, stateTransition, immediateValue)


def test_reference_style_driver_cash(S, oracle):
    """Reads like src/cash/singleItem/CashConstraint.java:91-146."""
    spec, init = cases.case_C_rich()
    recursion = S.CashRecursion(spec)
    recursion.setTreeMapCacheAction()
    s0 = S.CashState(1, *init[0])
    rows, iv, _ = oracle.topdown(spec, init[:1])
    assert recursion.getExpectedValue(s0) == iv[0]
    assert recursion.getAction(s0) == rows[0][-2]
    assert np.array_equal(recursion.getOptTable(), rows[:, :4])


def test_reference_style_driver_two_product(S, oracle):
    """Reads like src/cash/multiItem/MultiItemCash.java:123-139 (commented-out solve block)."""
    spec, init = cases.case_M2_small()
    recursion = S.CashRecursionMulti(spec)
    iniState = S.CashStateMulti(1, *init[0])
    rows, iv, _ = oracle.topdown(spec, init)
    assert recursion.getExpectedValue(iniState) == iv[0]
    n = spec.max_order_idx + 1
    first = rows[0]
    assert recursion.getAction(iniState) == S.Actions(int(first[-2]) // n, int(first[-2]) % n)


def test_two_product_tolerance_changes_the_answer(S, oracle):
    """`> val + 0.1` is not a plain maximum: with the tolerance switched off the policy differs somewhere,
    and both variants match the oracle."""
    spec, _ = cases.case_M2_small()
    Va, Qa, _, _ = oracle.dense(spec)
    spec0, _ = cases.case_M2_small()
    spec0.tie_tolerance = 0.0
    Vb, Qb, _, _ = oracle.dense(spec0)
    assert not np.array_equal(Qa, Qb)
    for sp, Vo, Qo in ((spec, Va, Qa), (spec0, Vb, Qb)):
        s, V, Q = _solve_all(S, sp)
        assert np.array_equal(V, Vo) and np.array_equal(Q, Qo)


def test_two_product_row_kernel(S, oracle):
    """The row-shared two-product kernel (integer prices): several cash segments per (inv1, inv2) pair with a
    ragged last segment, gamma < 1, non-integer salvage (last period only), demand lists that are not product
    grids; whole grid against the oracle, the thread-per-state kernel and sharded handles.  Non-integer
    prices must fall back to the thread-per-state kernel."""
    rng = np.random.default_rng(11)
    for cash_max, qb, inv_max, price, vc, sal, gamma in ((300, 5, 6, (4, 9), (2, 4), (1, 1.5), 0.95),
                                                        (131, 7, 4, (6, 5), (3, 1), (0.5, 2), 1.0),
                                                        (127, 3, 5, (3, 8), (1, 2), (1, 1), 1.0)):
        rows = []
        for _ in range(3):
            n = int(rng.integers(3, 9))
            d = np.stack([rng.integers(0, 6, n), rng.integers(0, 5, n)], axis=1).astype(float)
            rows.append(np.column_stack([d, rng.dirichlet(np.ones(n))]))
        spec = S.two_product_cash_model(rows, price=price, vari_cost=vc, salvage=sal, q_bound=qb, inv_max=inv_max,
                                        cash_min=0, cash_max=cash_max, gamma=gamma)
        Vo, Qo, evals, _ = oracle.dense(spec)
        s, V, Q = _solve_all(S, spec)
        assert s.stats()["kernel_used"] == S.KERNEL_TWO_PRODUCT_ROW and s.stats()["evals"] == evals
        assert np.array_equal(V, Vo) and np.array_equal(Q, Qo)
        g, Vg, Qg = _solve_all(S, spec, kernel=S.KERNEL_GENERIC)
        assert g.stats()["kernel_used"] == S.KERNEL_GENERIC
        assert np.array_equal(Vg, Vo) and np.array_equal(Qg, Qo)
    spec = S.two_product_cash_model(rows, price=(4.5, 9), vari_cost=(2, 4), salvage=(1, 1), q_bound=4, inv_max=5,
                                    cash_min=0, cash_max=60)
    Vo, Qo, _, _ = oracle.dense(spec)
    s, V, Q = _solve_all(S, spec)
    assert s.stats()["kernel_used"] == S.KERNEL_GENERIC
    assert np.array_equal(V, Vo) and np.array_equal(Q, Qo)


def test_reference_style_driver_workforce(S, oracle):
    """Reads like src/workforce/WorkforcePlanning.java:106-118."""
    spec, init = cases.case_W_small()
    recursion = S.StaffRecursion(spec)
    initialState = S.StaffState(1, 0)
    rows, iv, _ = oracle.topdown(spec, init)
    assert recursion.getExpectedValue(initialState) == iv[0]
    assert recursion.getAction(initialState) == int(rows[0][-2])


def test_reference_style_driver_survival(S, oracle):
    spec, init = cases.case_F_small()
    recursion = S.RiskRecursion(spec)
    s0 = S.RiskState(1, init[0][0], init[0][1], False)
    rows, iv, _ = oracle.topdown(spec, init)
    assert recursion.getSurvProb(s0) == iv[0]
    assert 0.0 <= iv[0] <= 1.0


# ---- full-size configurations ----------------------------------------------------------------
def _sample_check(S, oracle, spec, s, n=48, seed=3):
    """Period-by-period inductive check on a sample: recompute V_t, Q_t on the CPU from the GPU's
    own V_{t+1} table and compare bits."""
    rng = np.random.default_rng(seed)
    idx = np.unique(np.concatenate([[0, s.n_states - 1], rng.integers(0, s.n_states, n)]))
    Vn = None
    for t in range(spec.T, 0, -1):
        V, Q = s.period_tables(t)
        vo, qo = oracle.step_states(spec, t, Vn, idx)
        assert np.array_equal(V[idx], vo), f"period {t}"
        assert np.array_equal(Q[idx], qo), f"period {t}"
        Vn = V


def test_config_c1_full(S, oracle):
    spec = S.configs.c1()
    Vo, Qo, evals, _ = oracle.dense(spec)
    for kernel in (S.KERNEL_GENERIC, S.KERNEL_AUTO):
        s, V, Q = _solve_all(S, spec, kernel=kernel)
        assert np.array_equal(V, Vo) and np.array_equal(Q, Qo)
        assert s.stats()["evals"] == evals == 133399266.0


def test_config_c2_full(S, oracle):
    spec = S.configs.c2()
    Vo, Qo, evals, _ = oracle.dense(spec)
    s, V, Q = _solve_all(S, spec)
    assert np.array_equal(V, Vo) and np.array_equal(Q, Qo)


def test_config_c3_sampled(S, oracle):
    spec = S.configs.c3(T=3)          # full 501 x 2001 grid, 3 of the 12 periods
    s = S.Solver(spec).solve()
    assert s.n_states == 1002501 and s.stats()["kernel_used"] == S.KERNEL_CASH_DIAG
    _sample_check(S, oracle, spec, s, n=24)
    for k in (S.KERNEL_GENERIC, S.KERNEL_CASH_INT):
        g = S.Solver(spec, kernel=k).solve()
        for t in (1, 2, 3):
            Va, Qa = s.period_tables(t)
            Vg, Qg = g.period_tables(t)
            assert np.array_equal(Va, Vg) and np.array_equal(Qa, Qg)


def test_config_c4_sampled(S, oracle):
    spec = S.configs.c4(T=3)          # full 1001 x 101 x 101 grid, 3 of the 20 periods
    s = S.Solver(spec).solve()
    assert s.n_states == 10211201
    _sample_check(S, oracle, spec, s, n=64)
    # V(x, q1, q2) depends on (x, q1) only through x + q1: an exact structural identity
    V, Q = s.period_tables(1)
    V3 = V.reshape(1001, 101, 101)
    assert np.array_equal(V3[100, 7, :], V3[107, 0, :]) and np.array_equal(V3[500, 50, :], V3[520, 30, :])
    # the folded solve and the generic kernel give the same tables as the staged brute-force kernel
    assert s.stats()["kernel_used"] in (S.KERNEL_LEAD_Q2, S.KERNEL_LEAD_Q2M)
    for kw in ({"dedup": True}, {"kernel": S.KERNEL_GENERIC}, {"kernel": S.KERNEL_STAGED}, {"kernel": S.KERNEL_LEAD_SLAB},
               {"kernel": S.KERNEL_LEAD_COL}):
        d = S.Solver(spec, **kw).solve()
        Vd, Qd = d.period_tables(1)
        assert np.array_equal(Vd, V) and np.array_equal(Qd, Q)


def test_config_c5_sampled(S, oracle):
    spec = S.configs.c5(n_states=1_000_000, T=2)
    s = S.Solver(spec).solve()
    _sample_check(S, oracle, spec, s, n=64)
    assert s.stats()["kernel_used"] == S.KERNEL_TILED2
    # the tiled variants and the generic kernel are independent implementations: whole-grid agreement
    for k in (S.KERNEL_GENERIC, S.KERNEL_TILED):
        g = S.Solver(spec, kernel=k).solve()
        for t in (1, 2):
            Va, Qa = s.period_tables(t)
            Vg, Qg = g.period_tables(t)
            assert np.array_equal(Va, Vg) and np.array_equal(Qa, Qg)


# ---- J1: the measured configurations at FULL size and FULL horizon -------------------------------
def _fullsize_golden(name):
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fullsize.json")
    if not os.path.exists(path):
        pytest.skip("tests/golden/fullsize.json not generated (tests/golden/make_fullsize_golden.py)")
    g = json.load(open(path))
    if name not in g:
        pytest.skip(f"{name} not in tests/golden/fullsize.json")
    return g[name]


def _golden_spec(spec, gold):
    """The hashes only mean something on the very pmf table the frozen oracle run used (the fixture carries it)."""
    assert gold["pmf_same_every_period"]
    row = np.asarray(gold["pmf"][0], dtype=np.float64)
    for r in spec.pmf:
        assert np.array_equal(row, np.asarray(r)), "pmf table differs from the one the golden run used"


def _hash_check(s, gold):
    """Whole grid, every period: SHA-256 of the float64 V_t and Q_t bytes against the frozen oracle run."""
    import hashlib
    assert s.n_states == gold["n_states"] and s.T == gold["T"]
    V = np.empty(s.n_states)
    Q = np.empty(s.n_states)
    for t in range(1, s.T + 1):
        s.period_tables(t, out_v=V, out_q=Q)
        assert hashlib.sha256(V.tobytes()).hexdigest() == gold["sha256_V"][t - 1], f"V, period {t}"
        assert hashlib.sha256(Q.tobytes()).hexdigest() == gold["sha256_Q"][t - 1], f"Q, period {t}"
    v, q = s.value(1, [gold["init"]])
    assert v[0] == float.fromhex(gold["V1_init"]) and q[0] == gold["Q1_init"]


def test_config_c3_full_horizon(S, oracle):
    """C3 exactly as benched: 1,002,501 states, T = 12.  Every period: inductive sample check against the
    oracle, and the whole grid against the frozen whole-grid oracle run."""
    spec = S.configs.c3()
    s = S.Solver(spec).solve()
    assert s.n_states == 1002501 and spec.T == 12
    assert s.stats()["kernel_used"] == S.KERNEL_CASH_DIAG
    _sample_check(S, oracle, spec, s, n=32)
    gold = _fullsize_golden("c3")
    _golden_spec(spec, gold)
    _hash_check(s, gold)
    assert s.stats()["evals"] == gold["evals"]


def test_config_c4_full_horizon(S, oracle):
    """C4 exactly as benched: 10,211,201 states, T = 20; brute force and folded."""
    spec = S.configs.c4()
    s = S.Solver(spec).solve()
    assert s.n_states == 10211201 and spec.T == 20
    assert s.stats()["kernel_used"] == S.KERNEL_LEAD_Q2M   # the full grid is an unsliced launch: shared products
    _sample_check(S, oracle, spec, s, n=64)
    gold = _fullsize_golden("c4")
    _golden_spec(spec, gold)
    _hash_check(s, gold)
    assert s.stats()["evals"] == gold["evals"]
    s.close()
    d = S.Solver(spec, dedup=True).solve()
    _hash_check(d, gold)


def test_config_c5_bench_grid_full_horizon(S, oracle):
    """The C5 point the round-1 bench line was quoted on: 1e7 states x 200 x 200, T = 4."""
    spec = S.configs.c5(n_states=10_000_000)
    s = S.Solver(spec).solve()
    assert s.stats()["kernel_used"] == S.KERNEL_TILED2
    _sample_check(S, oracle, spec, s, n=64)
    gold = _fullsize_golden("c5_1e7")
    _golden_spec(spec, gold)
    _hash_check(s, gold)
    assert s.stats()["evals"] == gold["evals"]


def test_config_c5_1e8_sampled(S, oracle):
    """The largest single-GPU point of the sweep (1e8 states, T = 4): inductive sample check of every period."""
    spec = S.configs.c5(n_states=100_000_000)
    s = S.Solver(spec).solve()
    _sample_check(S, oracle, spec, s, n=48)


# ---- the reference's own recorded outputs, on the GPU ---------------------------------------------------------------
def _multi_pmf(vals1, probs1, vals2, probs2, T):
    """GetPmfMulti.getPmf for DiscreteDistribution (GetPmfMulti.java:158-171): all pairs, product 1 outermost."""
    rows = np.array([(a, b, pa * pb) for a, pa in zip(vals1, probs1) for b, pb in zip(vals2, probs2)], dtype=float)
    return [rows.copy() for _ in range(T)]


def test_multilead_reference_record_T2(S, oracle):
    """src/cash/overdraft/MultiProductLeadtime.java:41-43, recorded by the reference's author: 'when T = 2, final
    optimal cash is -17.800000000000008, optimal order quantity in the first period is: Q1 = 40, Q2 = 20'.
    The GPU's reached-state solve (sdpb_reached_solve) reproduces the Java program's printed output to the last
    digit, and agrees with the CPU oracle's restatement of the same loop."""
    vals = ([20, 30, 40], [10, 15, 20])
    probs = ([0.25, 0.5, 0.25], [0.25, 0.5, 0.25])
    recursion = S.CashRecursionMultiLead(_multi_pmf(vals[0], probs[0], vals[1], probs[1], 2), Qbound=50)
    iniState = S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0)
    finalValue = 0.0 + recursion.getExpectedValue(iniState)          # iniCash + recursion.getExpectedValue(iniState), :236
    assert finalValue == -17.800000000000008
    act = recursion.getAction(iniState)
    assert (act.getFirstAction(), act.getSecondAction()) == (40, 20)
    v, q1, q2, ns = oracle.multi_lead(2, 50, vals[0], probs[0], vals[1], probs[1])
    assert (finalValue, 40, 20) == (v, q1, q2) and sum(recursion.n_states) == ns


@pytest.mark.parametrize("T,qb,ovh", [(3, 7, 100.0), (3, 9, 20.0), (4, 4, 35.0), (1, 12, 100.0)])
def test_multilead_matches_oracle(T, qb, ovh, S, oracle):
    """Horizons and action bounds the CPU oracle solves in seconds: value, first-period actions and the number of
    visited states must equal the literal top-down recursion's."""
    vals = ([10, 30], [5, 15])
    probs = ([0.5, 0.5], [0.5, 0.5])
    rec = S.CashRecursionMultiLead(_multi_pmf(vals[0], probs[0], vals[1], probs[1], T), Qbound=qb, overheadCost=[ovh] * T)
    st = S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0)
    v = rec.getExpectedValue(st)
    vo, q1, q2, ns = oracle.multi_lead(T, qb, vals[0], probs[0], vals[1], probs[1], overhead=ovh)
    act = rec.getAction(st)
    assert v == vo and (act.getFirstAction(), act.getSecondAction()) == (q1, q2)
    assert sum(rec.n_states) == ns


@pytest.mark.parametrize("T,qb,cash", [(2, 8, 0.0), (2, 12, 25.0), (3, 5, 10.0), (1, 10, 30.0)])
def test_multi_xr_matches_oracle(T, qb, cash, S, oracle):
    """CashRecursionMultiXR with the MultiItemCashXR.java lambdas (Poisson demand through GetPmfMulti, `(int)` casts,
    state (x1, x2, R)) over the reached states: value, first-period order-up-to levels and the number of visited states
    equal the oracle's literal top-down recursion."""
    pmf = S.GetPmfMulti([[S.PoissonDist(4)] * T, [S.PoissonDist(3)] * T], 0.99, 1).tables()
    rec = S.CashRecursionMultiXR(pmf, price=(5, 10), variCost=(1, 2), Qbound=qb, maxInventoryState=40, maxCashState=500)
    st = S.CashStateMultiXR(1, 0, 0, cash)
    v = rec.getExpectedValue(st)
    vo, a1, a2, ns = oracle.reached(1, pmf, qb, (5, 10), (1, 2), (0.5, 1.0), [0, 0, cash], max_inv=40, max_cash=500)
    assert v == vo and rec.getAction(st) == [a1, a2]
    assert sum(rec.n_states) == ns


@pytest.mark.parametrize("T,qb,cash,dr", [(2, 8, 10.0, 0.0), (2, 12, 25.0, 0.05), (3, 5, 14.0, 0.0), (1, 10, 30.0, 0.0)])
def test_cash_recursion_v_matches_oracle(T, qb, cash, dr, S, oracle):
    """CashRecursionV (V / Pi form, the boundary function boundFinalCash valuing the states of period T+1, affordable
    order-up-to pairs, `> val + 0.01`) with the MultiItemYR.java lambdas, over the reached states."""
    pmf = S.GetPmfMulti([[S.PoissonDist(4)] * T, [S.PoissonDist(3)] * T], 0.99, 1).tables()
    rec = S.CashRecursionV(pmf, price=(5, 10), variCost=(1, 2), depositeRate=dr, Qbound=qb, maxInventoryState=40,
                           maxCashState=500)
    st = S.CashStateMulti(1, 0, 0, cash)
    v = rec.getExpectedValueV(st)
    vo, a1, a2, ns = oracle.reached(2, pmf, qb, (5, 10), (1, 2), (0.5, 1.0), [0, 0, cash], deposit_rate=dr, max_inv=40,
                                    max_cash=500)
    assert v == vo and rec.getAction(st) == [a1, a2]
    assert sum(rec.n_states) == ns


@pytest.mark.parametrize("means,K,cash,rate", [((6, 3, 2, 5), 8.0, 33.0, 0.0), ((20, 7, 2, 14), 24.0, 33.0, 0.0),
                                               ((5, 4, 6), 0.0, 27.0, 0.1)])
def test_cash_constraint_test_lambdas(means, K, cash, rate, S, oracle):
    """src/cash/singleItem/CashConstraintTest.java:76-116 -- the one single-product driver whose states do not sit on a
    grid: inventory and cash are rounded as Math.round(v * 0.1) / 0.1 (30.000000000000004 ...) and the initial cash, 33,
    is not a rounded value at all.  Solved over the reached states; reads like the driver's :121-129."""
    dists = [S.PoissonDist(m) for m in means]
    pmf = S.GetPmf(dists, 0.9999, 1).getpmf()
    recursion = S.CashRecursionRounded(pmf, price=4, variCost=1, fixOrderCost=K, holdingCost=0, salvageValue=0.5,
                                       interestRate=rate, minCashRequired=0, maxOrderQuantity=60, maxInventoryState=500,
                                       minCashState=-100, maxCashState=2000)
    initialState = S.CashState(1, 0, cash)
    finalValue = cash + recursion.getExpectedValue(initialState)
    vo, a1, _, ns = oracle.reached(3, pmf, 61, (4, 0), (1, 0), (0.5, 0), [0, 0, cash], deposit_rate=rate, min_inv=0,
                                   max_inv=500, min_cash=-100, max_cash=2000, fixed_cost=K, state_q=0.1)
    assert finalValue == cash + vo and recursion.getAction(initialState) == a1
    assert sum(recursion.n_states) == ns and recursion.n_states[0] == 1


def test_multilead_reference_record_T3_three_point(S):
    """src/cash/overdraft/MultiProductLeadtime.java:35-39 -- the third output the reference's author recorded: 3 periods,
    demands {20,30,40} x {10,15,20} with probabilities {.25,.5,.25}: 'final optimal cash is 91.19499999999998 ... Q1 = 40,
    Q2 = 20 ... running time is 2863.0s'.  1.78e7 reached states; about 1.6 s on the device."""
    rec = S.CashRecursionMultiLead(_multi_pmf([20, 30, 40], [0.25, 0.5, 0.25], [10, 15, 20], [0.25, 0.5, 0.25], 3),
                                   Qbound=50)
    st = S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0)
    finalValue = 0.0 + rec.getExpectedValue(st)
    act = rec.getAction(st)
    assert finalValue == 91.19499999999998
    assert (act.getFirstAction(), act.getSecondAction()) == (40, 20)
    assert rec.n_states == [1, 2500, 17772500]


def test_multilead_reference_record_T3_no_overhead(S):
    """src/cash/overdraft/MultiProductLeadtime.java:30 -- 'final optimal cash is 441.57499999999993 for overhead cost 0'
    (3 periods, the three-point demands).  The two other figures of that older comment line (91.26875 and
    272.23749999999995 for overhead 100 and 50) come from parameters the comment does not state: the author's own later
    run of the overhead-100 instance (:37) prints 91.19499999999998 -- reproduced above -- and with overhead 50 this library
    gives 272.254375."""
    pmf = _multi_pmf([20, 30, 40], [0.25, 0.5, 0.25], [10, 15, 20], [0.25, 0.5, 0.25], 3)
    rec = S.CashRecursionMultiLead(pmf, Qbound=50, overheadCost=[0.0] * 3)
    st = S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0)
    assert 0.0 + rec.getExpectedValue(st) == 441.57499999999993
    act = rec.getAction(st)
    assert (act.getFirstAction(), act.getSecondAction()) == (40, 20)


def test_multilead_reference_record_T3(S):
    """src/cash/overdraft/MultiProductLeadtime.java:45-50 -- the live code of the reference: 3 periods, demands
    {10,30} x {5,15}: 'final optimal cash is -76.56 ... Q1 = 30, Q2 = 15 ... running time is 1568.0s'.  1.7e7 states and
    1.7e11 evaluations; the CPU oracle needs 34 minutes for it (tests/test_oracle.py, opt-in), the GPU about a second."""
    rec = S.CashRecursionMultiLead(_multi_pmf([10, 30], [0.5, 0.5], [5, 15], [0.5, 0.5], 3), Qbound=50)
    st = S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0)
    finalValue = 0.0 + rec.getExpectedValue(st)
    act = rec.getAction(st)
    assert finalValue == -76.56                             # Double.toString prints the shortest digits that identify the double
    assert (act.getFirstAction(), act.getSecondAction()) == (30, 15)
    assert rec.n_states[0] == 1 and sum(rec.n_states) > 1.6e7
    print(f"multilead T=3: {rec.n_states} states, {rec.solve_ms:.0f} ms on the device")
