"""The row-shared cash kernels, bi_cash_tail<KIND, MODE, PEN, DIV> and bi_cash_row<SURV, MIN>, at every template
instantiation and at the edges of the host plans that admit a model to them (plan_cash_tail and cash_row_ok in
kernel_cash.cuh).  Their speed comes from strength reductions that are exact only inside those plans (the cash clamp
behind Math.round, Java's long division by multiply and shift, +0.0 terms skipped, one action count per 128-level CTA),
so a plan that admits a model it should refuse writes a wrong table without any error.

Every model is solved three ways and compared whole grid, every period, with ==: the kernel under test against the CPU
oracle (values, order quantities and the evaluation count), the generic kernel against the oracle, and the kernel the
solve reports against the one the case names."""
import os

import numpy as np
import pytest

import cases
import test_fuzz_gpu as fuzz
import sdpb200 as S
from sdpb200 import abi as A

pytestmark = pytest.mark.gpu

DEP, OD, ODL, ODT = A.COST_CASH_DEPOSIT, A.COST_CASH_OVERDRAFT, A.COST_CASH_OD_LIMIT, A.COST_CASH_OD_TESTING
KINDS = (DEP, OD, ODL, ODT)
TAIL, ROW, GENERIC = S.KERNEL_CASH_TAIL, S.KERNEL_CASH_ROW, S.KERNEL_GENERIC

# per kind: the factory and parameters that switch every term of its lambda on
_FACTORY = {
    DEP: (S.cash_constraint_model, dict(price=5.5, vari_cost=1.25, fixed_cost=1.0, hold_cost=0.25, salvage=0.5,
                                        overhead=1.5, deposit_rate=0.0625)),
    OD: (S.cash_overdraft_model, dict(price=6.0, vari_cost=1.5, fixed_cost=2.0, salvage=0.75, r0=0.0625, r2=0.125,
                                      r3=1.5, od_limit=6.0, interest_free=1.0)),
    ODL: (S.cash_overdraft_limit_model, dict(price=6.0, vari_cost=1.5, fixed_cost=1.0, hold_cost=0.25, salvage=0.5,
                                             interest_rate=0.125, deposit_rate=0.0625)),
    ODT: (S.cash_overdraft_testing_model, dict(price=6.5, vari_cost=1.5, fixed_cost=1.0, hold_cost=0.25,
                                               interest_rate=0.2, min_cash_required=-2.0)),
}


def model(kind, pmf, q=(A.Q_DIV, 10.0, 10.0), cash=(-8.0, 19.0), direction=None, terminal=False, attrs=None, **kw):
    """A model of `kind` with the parameters of _FACTORY overridden by `kw`; `attrs` are set on the spec afterwards
    (per-period arrays the factory does not take); `terminal` adds a boundary table."""
    fn, base = _FACTORY[kind]
    args = dict(base, inv_min=0.0, inv_max=9.0, max_order=7, quantiser=q[0], q_mul=q[1], q_div=q[2],
                cash_min=cash[0], cash_max=cash[1])
    if kind in (OD, ODL):
        args["overhead_t"] = [1.5] * len(pmf)
    args.update(kw)
    spec = fn(pmf, **args)
    for k, v in (attrs or {}).items():
        setattr(spec, k, v)
    if direction is not None:
        spec.direction = direction
    if terminal:
        spec.terminal_value = spec.tabulate(lambda x, w: 0.5 * w + 0.75 * x - 0.125 * np.maximum(-w, 0.0))
    spec.name = f"kind{kind}"
    return spec


def _check(spec, oracle, runs=((S.KERNEL_AUTO, TAIL),), tag=""):
    """`runs`: (requested kernel, kernel the solve must report) pairs; the generic kernel is always added.  Whole grid,
    every period, == against the oracle; returns the kernels the solves reported."""
    Vo, Qo, evals, _ = oracle.dense(spec)
    reported = []
    for kernel, want in tuple(runs) + ((GENERIC, GENERIC),):
        with S.Solver(spec, kernel=kernel) as s:
            s.solve()
            st = s.stats()
            for t in range(1, spec.T + 1):
                V, Q = s.period_tables(t)
                bad = np.flatnonzero((V != Vo[t - 1]) | (Q != Qo[t - 1]))
                assert len(bad) == 0, (f"{tag} {spec.name} kernel={kernel} ran {st['kernel_used']} t={t}: {len(bad)} "
                                       f"states differ, first {[s.state_of_index(int(i)).tolist() for i in bad[:3]]} "
                                       f"V {V[bad[:3]]} vs {Vo[t - 1][bad[:3]]}, Q {Q[bad[:3]]} vs {Qo[t - 1][bad[:3]]}")
            assert st["evals"] == evals, (tag, spec.name, kernel)
            assert want is None or st["kernel_used"] == want, (tag, spec.name, kernel, st["kernel_used"], want)
            reported.append(st["kernel_used"])
    return reported


def _signed_unit_cost(spec):
    """A cash-limited action set with a unit cost whose sign bit is set: the bound falls as cash grows."""
    vs = spec.vari_cost_t if spec.vari_cost_t is not None else [spec.vari_cost] * spec.T
    return bool(spec.flags & A.F_CASH_LIMITED_ACTIONS) and any(np.signbit(v) for v in vs)


# ---- a. every instantiation ---------------------------------------------------------------------------------------
def tail_key(spec, t):
    """The bi_cash_tail<KIND, MODE, PEN, DIV> that launch_cash_tail picks for period t."""
    mode = 0 if t < spec.T else (2 if spec.terminal_value is not None else 1)
    pen = spec.cost_kind == DEP and spec.penalty_cost != 0.0
    div = spec.quantiser == A.Q_LONGDIV and int(spec.q_div) != 1
    return spec.cost_kind, mode, pen, div


def row_key(spec):
    """The bi_cash_row<SURVIVAL, IS_MIN> that launch_cash_row picks."""
    return spec.recursion == A.REC_SURVIVAL, spec.recursion != A.REC_SURVIVAL and spec.direction == A.MIN


ALL_TAIL_KEYS = {(k, mode, pen, div) for k in KINDS for mode in (0, 1, 2) for pen in ((False, True) if k == DEP else (False,))
                 for div in (False, True)}


def coverage_models():
    """Two-period models (periods 1 and T) over kind x DIV x PEN x boundary table.  Their demand rows are far inside the
    plan's shared-memory limit, the only per-period input of plan_cash_tail, so every period of a model the plan admits
    runs bi_cash_tail."""
    out, n = [], 0
    for kind in KINDS:
        for div in (False, True):
            for pen in ((0.0, 0.5) if kind == DEP else (0.0,)):
                for terminal in (False, True):
                    if div:   # Java long division by 10 or by 2 after rounding
                        q, cash = ((A.Q_LONGDIV, 10.0, 10.0), (-40.0, 160.0)) if terminal else ((A.Q_LONGDIV, 2.0, 2.0), (-40.0, 160.0))
                    else:     # the 0.1 grid, or round(w*1)/1
                        q, cash = ((A.Q_DIV, 10.0, 10.0), (-8.0, 19.0)) if terminal else ((A.Q_LONGDIV, 1.0, 1.0), (-40.0, 160.0))
                    kw = dict(penalty_cost=pen) if kind == DEP else {}
                    out.append(model(kind, cases.pmf([4, 5], 0.99), q=q, cash=cash, terminal=terminal,
                                     direction=A.MIN if n % 2 else A.MAX, gamma=0.95 if n % 3 == 1 else 1.0, **kw))
                    n += 1
    return out


def test_every_cash_tail_instantiation(oracle):
    keys = set()
    for spec in coverage_models():
        _check(spec, oracle, tag="coverage")
        keys |= {tail_key(spec, t) for t in range(1, spec.T + 1)}
    assert len(ALL_TAIL_KEYS) == 30
    assert keys == ALL_TAIL_KEYS, f"{len(keys & ALL_TAIL_KEYS)}/30 bi_cash_tail keys, missing {ALL_TAIL_KEYS - keys}"


def test_every_cash_row_instantiation(oracle):
    pmf = cases.pmf([4, 5, 4], 0.99)
    jobs = [(S.cash_survival_model(pmf, price_t=[4.5, 5.0, 4.0], vari_cost_t=[1.0, 1.5, 2.0], overhead_t=[3.0, 2.0, 4.0],
                                   hold_cost=0.25, max_order=9, inv_min=0, inv_max=9, cash_min=-10, cash_max=150),
             ((S.KERNEL_AUTO, ROW),))]
    for direction in (A.MIN, A.MAX):   # the expectation recursion runs bi_cash_row on request
        jobs.append((model(DEP, pmf, direction=direction, penalty_cost=0.5), ((ROW, ROW), (S.KERNEL_AUTO, TAIL))))
    keys = set()
    for spec, runs in jobs:
        _check(spec, oracle, runs, tag="row coverage")
        keys.add(row_key(spec))
    assert keys == {(True, False), (False, True), (False, False)}, f"{len(keys)}/3 bi_cash_row keys"


# ---- b. segment geometry --------------------------------------------------------------------------------------------
def geometry_model(kind, nW, direction, gamma):
    """nW levels of the 0.1 grid from -3.0; the cash-limited action count rises from 1 to the maximum (9) over three
    cash levels inside one 128-level segment, the middle one of the grid."""
    seg = ((nW - 1) // 2) // 128
    lt = seg * 128 + min(64, (nW - seg * 128) // 2)          # first lane with more than one action
    reserve = (-30 + lt) / 10.0 - 0.05                       # (w - reserve) / 0.03 = 1.67, 5, 8.3 on lanes lt, lt+1, lt+2
    cash = (-3.0, (-30 + nW - 1) / 10.0)
    common = dict(cash=cash, vari_cost=0.03, fixed_cost=0.5, max_order=8, inv_max=4.0, direction=direction, gamma=gamma)
    if kind == DEP:
        return model(DEP, cases.pmf([3, 4], 0.99), overhead=reserve - 0.5, **common)
    return model(ODT, cases.pmf([3, 4], 0.99), min_cash_required=reserve - 0.5, **common)


@pytest.mark.parametrize("nW", [1, 2, 127, 128, 129, 255, 256, 257, 385])
def test_segment_geometry(nW, oracle):
    for i, (direction, gamma) in enumerate(((A.MAX, 1.0), (A.MIN, 0.9))):
        spec = geometry_model(DEP, nW, direction, gamma)
        assert oracle.grid(spec)[0] == 5 * nW
        _check(spec, oracle, ((S.KERNEL_AUTO, TAIL), (ROW, ROW)), tag=f"nW={nW}")
        spec = geometry_model(ODT, nW, (A.MIN, A.MAX)[i], gamma)
        _check(spec, oracle, tag=f"nW={nW}")


# ---- c. plan edges ----------------------------------------------------------------------------------------------------
def tail_bound(spec):
    """plan_cash_tail's bound on |w'|, term for term and in the same order."""
    price, v, ovh = abs(spec.price), abs(spec.vari_cost), abs(spec.overhead)
    for t in range(spec.T):
        price = max(price, abs(spec.price_t[t] if spec.price_t is not None else spec.price))
        if spec.vari_cost_t is not None:
            v = max(v, abs(spec.vari_cost_t[t]))
        if spec.overhead_t is not None:
            ovh = max(ovh, abs(spec.overhead_t[t]))
    dmax = max(abs(float(d)) for r in spec.pmf for d in np.asarray(r)[:, 0])
    stock = max(abs(spec.inv_min), abs(spec.inv_max)) + float(spec.max_order_idx) * spec.step
    cash = max(abs(spec.cash_min), abs(spec.cash_max))
    rates = 1.0 + abs(spec.deposit_rate) + abs(spec.r0) + abs(spec.r2) + abs(spec.r3) + abs(spec.penalty_cost)
    return ((cash + abs(spec.fixed_cost) + v * spec.max_order_idx * spec.step + ovh + abs(spec.od_limit) +
             abs(spec.interest_free)) * rates * rates +
            (price + abs(spec.salvage) + abs(spec.hold_cost)) * (stock + dmax) * rates)


def test_magnitude_guard_edge(oracle):
    """bound * |q_mul| < 2^30, with q_mul = 10 and prices of a few million: Math.round sees |w' * 10| of about 2^28
    before the clamp.  The price one unit below the edge runs bi_cash_tail, one unit above does not."""
    pmf = cases.pmf([4, 5], 0.99)
    for kind in KINDS:
        q = (A.Q_DIV, 10.0, 10.0) if kind in (DEP, ODT) else (A.Q_LONGDIV, 10.0, 10.0)

        def at(p):
            return model(kind, pmf, q=q, price=float(p))
        probe = at(0.0)
        per_unit = (tail_bound(at(1000.0)) - tail_bound(probe)) / 1000.0
        p = int((2 ** 30 / 10 - tail_bound(probe)) / per_unit)
        while tail_bound(at(p)) * 10 >= 2 ** 30:
            p -= 1
        while tail_bound(at(p + 1)) * 10 < 2 ** 30:
            p += 1
        inside, outside = at(p), at(p + 1)
        assert tail_bound(inside) * 10 < 2 ** 30 <= tail_bound(outside) * 10 and p > 1e6
        _check(inside, oracle, tag=f"price {p}")
        _check(outside, oracle, ((S.KERNEL_AUTO, ROW if kind == DEP else GENERIC),), tag=f"price {p + 1}")


@pytest.mark.parametrize("q_div", [2, 3, 7, 10, 1000])
def test_multiply_shift_edge(q_div, oracle):
    """Java's long division by multiply and shift is exact for |kk| < q_div * 2^16; the plan bounds the clamped
    integer by round(cash_min * q_mul) and round(cash_max * q_mul).  Both bounds one inside the limit, then the upper
    and the lower one on it (division truncates toward zero, so the negative side has its own edge)."""
    lim = q_div << 16
    pmf = cases.pmf([2, 3], 0.9)
    kind = KINDS[[2, 3, 7, 10, 1000].index(q_div) % 4]
    refused = ROW if kind == DEP else GENERIC
    for cash, used in (((-(lim - 1), lim - 1), TAIL), ((-(lim - 1), lim), refused), ((-lim, lim - 1), refused)):
        spec = model(kind, pmf, q=(A.Q_LONGDIV, 1.0, float(q_div)), cash=(float(cash[0]), float(cash[1])),
                     inv_max=1.0, max_order=3)
        _check(spec, oracle, ((S.KERNEL_AUTO, used),), tag=f"q_div={q_div} cash={cash}")


def test_magic_constant_range(oracle):
    """q_magic = ceil(2^47 / q_div) exists for q_div < 2^15 only; at 32768 the plan must refuse."""
    pmf = cases.pmf([3, 4], 0.99)
    for q_div in (32767, 32768):
        for kind in (DEP, OD):
            spec = model(kind, pmf, q=(A.Q_LONGDIV, 10000.0, float(q_div)), cash=(-30.0, 30.0))
            used = TAIL if q_div < 32768 else (ROW if kind == DEP else GENERIC)
            _check(spec, oracle, ((S.KERNEL_AUTO, used),), tag=f"q_div={q_div}")


def _wide_pmf(sizes, seed):
    rng = np.random.default_rng(seed)
    return [np.stack([np.arange(n, dtype=float), rng.dirichlet(np.ones(n))], axis=1) for n in sizes]


@pytest.mark.parametrize("D", [1024, 1025, 2048, 2049])
def test_shared_memory_edge(D, oracle):
    """48 bytes of shared memory per demand point: 1024 points fit the default 48 KB, 1025 need the opt-in attribute,
    2048 fill the plans' 96 KB and 2049 go to the generic kernel."""
    fits = D <= 2048
    for kind in (DEP, ODL):
        spec = model(kind, _wide_pmf([D, D], D), cash=(-2.0, 10.0), inv_max=3.0, max_order=3)
        runs = [(S.KERNEL_AUTO, TAIL if fits else GENERIC)]
        if kind == DEP:
            runs.append((ROW, ROW if fits else GENERIC))
        _check(spec, oracle, runs, tag=f"D={D}")


def test_shared_memory_edge_inside_one_model(oracle):
    """Period 1 has 2048 demand points (bi_cash_tail), period 2 has 2049 (the generic kernel)."""
    for kind in (DEP, OD):
        spec = model(kind, _wide_pmf([2048, 2049], 7), cash=(-2.0, 10.0), inv_max=3.0, max_order=3)
        _check(spec, oracle, tag="D=2048|2049")


def test_price_and_overhead_rate_edges(oracle):
    """A price of +0.0 is admitted (revenue stays +0.0), a negative one is not; a deposit model's overhead rate up to 1."""
    pmf = cases.pmf([4, 5, 4], 0.99)
    jobs = []
    for kind in (DEP, ODL):
        refused = ROW if kind == DEP else GENERIC
        jobs += [(model(kind, pmf, attrs=dict(price_t=[4.5, 0.0, 3.0])), TAIL),
                 (model(kind, pmf, attrs=dict(price_t=[4.5, -0.5, 3.0])), refused)]
    jobs += [(model(DEP, pmf, overhead_rate=1.0), TAIL), (model(DEP, pmf, overhead_rate=1.0625), ROW)]
    for spec, used in jobs:
        _check(spec, oracle, ((S.KERNEL_AUTO, used),), tag=f"price_t={spec.price_t} rho={spec.overhead_rate}")


# ---- d. signs and zeros ---------------------------------------------------------------------------------------------
def _survival(v_t):
    return S.cash_survival_model(cases.pmf([5, 6, 4], 0.99), price_t=[4.5, 5, 4], vari_cost_t=v_t, overhead_t=[11, 9, 12],
                                 salvage=0.5, hold_cost=0.25, max_order=12, inv_min=0, inv_max=12, cash_min=-20, cash_max=150)


_PMF2 = cases.pmf([4, 5], 0.99)
# id: (model, kernel AUTO runs, kernel a bi_cash_row request runs or None); the reserve 2.5 is a grid point
UNIT_COST_CASES = {
    "C_plus_zero": (lambda: model(DEP, _PMF2, vari_cost=0.0, overhead=2.5, fixed_cost=0.0, cash=(-3.0, 12.7)), TAIL, ROW),
    "C_minus_zero": (lambda: model(DEP, _PMF2, vari_cost=-0.0, overhead=2.5, fixed_cost=0.0, cash=(-3.0, 12.7)), GENERIC, GENERIC),
    # the top lane of the first segment (w = -7.3) allows 8 actions, the lanes below w = -12 allow 13
    "C_negative": (lambda: S.cash_constraint_model(_PMF2, vari_cost=-1, max_order=12, inv_max=6, cash_min=-20, cash_max=60),
                   GENERIC, GENERIC),
    "C_mixed_signs": (lambda: model(DEP, _PMF2, attrs=dict(vari_cost_t=[1.25, -0.75])), GENERIC, GENERIC),
    "F_mixed_signs": (lambda: _survival([1.0, -0.5, 2.0]), GENERIC, GENERIC),
    "F_minus_zero": (lambda: _survival([1.0, -0.0, 2.0]), GENERIC, GENERIC),
    "DT_plus_zero": (lambda: model(ODT, _PMF2, vari_cost=0.0, min_cash_required=2.5, fixed_cost=0.0, cash=(-3.0, 12.7)),
                     TAIL, None),
    "DT_negative": (lambda: model(ODT, _PMF2, vari_cost=-0.5), GENERIC, None),
    # no cash-limited action set: a negative unit cost is only a number
    "D_negative": (lambda: model(OD, _PMF2, vari_cost=-1.0), TAIL, None),
    "DL_minus_zero": (lambda: model(ODL, _PMF2, vari_cost=-0.0), TAIL, None),
}


@pytest.mark.parametrize("case", list(UNIT_COST_CASES))
def test_unit_cost_signs(case, oracle):
    """The cash-limited bound max(0, ((w - reserve) - reserve2) / v) grows with w for v > 0 and v = +0.0 (inf above the
    reserve, NaN on it: one action, as in the oracle) and falls for v < 0 or v = -0.0, so the row kernels, which give
    a CTA the action count of its richest lane, must not take such models."""
    build, used, row_used = UNIT_COST_CASES[case]
    spec = build()
    runs = [(S.KERNEL_AUTO, used)] + ([(ROW, row_used)] if row_used is not None else [])
    _check(spec, oracle, runs, tag=case)
    assert (used == GENERIC) == _signed_unit_cost(spec)


def test_negative_zeros_and_degenerate_cash_axes(oracle):
    pmf = cases.pmf([4, 5], 0.99)
    jobs = [model(DEP, pmf, penalty_cost=-0.0, salvage=-0.0, hold_cost=-0.0),
            model(DEP, pmf, price=-0.0),
            model(ODL, pmf, salvage=-0.0, hold_cost=-0.0),
            model(OD, pmf, salvage=-0.0, fixed_cost=-0.0),
            model(DEP, pmf, cash=(2.5, 20.0)),                 # cash_min > 0
            model(ODT, pmf, cash=(1.0, 14.0)),
            model(DEP, pmf, cash=(7.5, 7.5)),                  # one cash level
            model(OD, pmf, cash=(-3.0, -3.0), q=(A.Q_LONGDIV, 10.0, 10.0)),
            # a 0.5 grid and .25-valued costs: w' * 2 ends in .5, on negative cash too (Math.round(-2.5) = -2)
            model(DEP, pmf, q=(A.Q_DIV, 2.0, 2.0), cash=(-12.0, 15.0), price=1.25, vari_cost=0.75, fixed_cost=0.5,
                  overhead=0.25, hold_cost=0.25, salvage=0.25, penalty_cost=0.25, deposit_rate=0.0),
            model(OD, pmf, q=(A.Q_LONGDIV, 2.0, 2.0), cash=(-12.0, 15.0), price=1.25, vari_cost=0.75, fixed_cost=0.25,
                  salvage=0.25, r0=0.0, r2=0.0, r3=0.0, interest_free=0.0, attrs=dict(overhead_t=[0.25, 0.75])),
            model(ODL, pmf, q=(A.Q_DIV, 2.0, 2.0), cash=(-12.0, 15.0), price=1.25, vari_cost=0.75, fixed_cost=0.25,
                  hold_cost=0.25, salvage=0.25, interest_rate=0.0, deposit_rate=0.0)]
    for spec in jobs:
        _check(spec, oracle, tag=f"{spec.cash_min}..{spec.cash_max}")


# ---- e. shards ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3, 5, 8])
def test_shards_cut_through_segments(world, oracle):
    pmf = cases.pmf([4, 5], 0.99)
    jobs = [(model(kind, pmf, cash=(-8.0, 19.0), terminal=kind == ODL), S.KERNEL_AUTO, TAIL) for kind in KINDS]
    jobs.append((model(DEP, pmf, cash=(-8.0, 19.0), direction=A.MIN), ROW, ROW))
    if world == 8:   # 5 states in 8 shards: three shards are empty
        jobs.append((model(DEP, pmf, cash=(1.0, 1.4), inv_max=0.0), S.KERNEL_AUTO, TAIL))
    for spec, kernel, used in jobs:
        Vo, Qo, evals, _ = oracle.dense(spec)
        with S.Group(spec, [0] * world, kernel=kernel) as g:
            g.solve()
            for t in range(1, spec.T + 1):
                V, Q = g.period_tables(t)
                assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), (spec.name, world, kernel, t)
            assert g.stats()["evals"] == evals
            ran = [sh.stats()["kernel_used"] for sh in g.shards if sh.grid.shard_hi > sh.grid.shard_lo]
            assert ran and all(k == used for k in ran), (spec.name, world, ran)
            if g.n_states < world:
                assert len(ran) < world


# ---- f. seeded fuzz -------------------------------------------------------------------------------------------------
_QUANTISERS = [(A.Q_DIV, 10.0, 10.0), (A.Q_DIV, 2.0, 4.0), (A.Q_DIV, 4.0, 2.0), (A.Q_LONGDIV, 1.0, 1.0),
               (A.Q_LONGDIV, 10.0, 10.0), (A.Q_LONGDIV, 10.0, 3.0), (A.Q_LONGDIV, 100.0, 7.0),
               (A.Q_LONGDIV, 1000.0, 1000.0), (A.Q_LONGDIV, 3.0, 2.0), (A.Q_LONGDIV, 1.0, 1000.0)]


def _signed(rng, x):
    r = rng.random()
    return -x if r < 0.2 else (-0.0 if r < 0.25 else x)


def fuzz_model(kind, rng):
    T = int(rng.integers(1, 4))
    pmf = fuzz._pmf(rng, T, int(rng.integers(1, 81)), gaps=rng.random() < 0.3)
    q = _QUANTISERS[int(rng.integers(len(_QUANTISERS)))]
    nW = int(rng.integers(1, 3001))
    span = (nW - 1) * (q[2] / q[1] if q[0] == A.Q_LONGDIV else 1.0 / q[2])
    lo = -float(np.round(span * rng.uniform(0, 0.6), 1))
    kw = dict(price=fuzz._cost(rng, False) + 0.5, vari_cost=_signed(rng, fuzz._cost(rng, False)),
              fixed_cost=fuzz._cost(rng, False), inv_min=float(rng.integers(0, 3)), max_order=int(rng.integers(0, 11)),
              gamma=float(rng.choice([1.0, 0.9])))
    kw["inv_max"] = kw["inv_min"] + float(rng.integers(0, 11))
    if kind == DEP:
        kw.update(hold_cost=fuzz._cost(rng, False), salvage=fuzz._cost(rng, False), overhead=fuzz._cost(rng, False),
                  overhead_rate=float(rng.choice([0, 0.125, 1.0])), deposit_rate=float(rng.choice([0, 0.25])),
                  penalty_cost=float(rng.choice([0, 0.5, 2.0])))
    elif kind == OD:
        kw.update(salvage=fuzz._cost(rng, False), r0=float(rng.choice([0, 0.125])), r2=0.125, r3=1.5,
                  od_limit=float(rng.integers(0, 30)), interest_free=float(rng.integers(0, 3)))
    elif kind == ODL:
        kw.update(hold_cost=fuzz._cost(rng, False), salvage=fuzz._cost(rng, False),
                  interest_rate=float(rng.choice([0.0, 0.125, 0.2])), deposit_rate=float(rng.choice([0, 0.0625])))
    else:
        kw.update(hold_cost=fuzz._cost(rng, False), interest_rate=float(rng.choice([0.0, 0.125, 0.2])),
                  min_cash_required=-float(rng.integers(0, 10)))
    attrs = {}
    if rng.random() < 0.5:
        attrs["price_t"] = [fuzz._cost(rng, False) + 0.5 for _ in range(T)]
        attrs["vari_cost_t"] = [_signed(rng, fuzz._cost(rng, False)) for _ in range(T)]
        attrs["overhead_t"] = [fuzz._cost(rng, False) for _ in range(T)]
        if kind == DEP:   # CashConstraint.java keeps the overhead back from ordering
            attrs["reserve_t"] = attrs["overhead_t"]
    return model(kind, pmf, q=q, cash=(lo, lo + span), direction=int(rng.integers(0, 2)),
                 terminal=rng.random() < 1 / 3, attrs=attrs, **kw)


@pytest.mark.parametrize("kind", KINDS, ids=["C", "D", "DL", "DT"])
def test_fuzz_row_shared_kinds(kind, oracle):
    rng = np.random.default_rng(1000 + kind)
    iters = int(os.environ.get("SDPB_FUZZ_ITERS", "40"))   # raise for a longer one-off campaign
    tail = 0
    for it in range(iters):
        spec = fuzz_model(kind, rng)
        runs = [(S.KERNEL_AUTO, None)] + ([(ROW, None)] if kind == DEP else [])
        reported = _check(spec, oracle, runs, tag=f"#{it}")
        used = reported[0]
        if _signed_unit_cost(spec):
            assert set(reported) == {GENERIC}, (it, reported, spec)
        else:
            assert used in (TAIL, ROW, GENERIC), (it, used)
        tail += used == TAIL
    assert tail >= iters // 2, f"only {tail} of {iters} models ran bi_cash_tail"
