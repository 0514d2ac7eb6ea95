"""The integer-exact cash kernels, bi_cash_diag<SURV, MIN> and bi_cash_int<SURV, MIN, LAST, R>, at every template
instantiation, sliced and unsliced, and at both sides of every edge of the host plans that admit a model to them
(plan_cash, cash_diag_ok, cash_int_shape and cash_diag_parts in kernel_cash.cuh).  Their speed comes from shortcuts that
are exact only inside those plans -- the diagonal register window, one running gather offset per 10-step block, the
shared stock-out entry, 16 cash levels per thread in the last period, action slices merged first-wins by
merge_action_slices -- so a plan that admits a model it should refuse writes a wrong table without any error.

Every model is solved whole grid, every period, and compared bit for bit with the CPU oracle (values, order quantities
and the evaluation count), once per requested kernel and once with the generic kernel.  A Python mirror of the host
shape functions predicts, per period, the kernel, its instantiation and its slice count; the solve must report the
kernel and the launch count (one per period, one more per sliced period) that the mirror predicts."""
import functools
import os

import numpy as np
import pytest

import sdpb200 as S
from sdpb200 import abi as A
from test_cash_row_kernels import tail_bound

pytestmark = pytest.mark.gpu

AUTO, GENERIC, DIAG, INT = S.KERNEL_AUTO, S.KERNEL_GENERIC, S.KERNEL_CASH_DIAG, S.KERNEL_CASH_INT
TAIL, ROW = S.KERNEL_CASH_TAIL, S.KERNEL_CASH_ROW
MAX, MIN = A.MAX, A.MIN


@functools.lru_cache(maxsize=None)
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- the mirror of the host plans -------------------------------------------------------------------------------------
def _small_int(x, lim=1048576.0):
    """cash_is_small_int"""
    return bool(np.floor(x) == x) and abs(x) < lim


def _per_period(spec, name, t):
    arr = getattr(spec, name + "_t")
    return float(arr[t]) if arr is not None else float(getattr(spec, name))


def dims(spec):
    """(nI, nW) of an integer grid (step 1, round(w*1)/1)."""
    return int(round(spec.inv_max - spec.inv_min)) + 1, int(round(spec.cash_max)) - int(round(spec.cash_min)) + 1


def plan_cash(spec):
    """Per period (price, v, ovh, d0) or None, term for term as plan_cash."""
    none = [None] * spec.T
    if spec.cost_kind != A.COST_CASH_DEPOSIT or spec.lead_time != 0 or spec.step != 1.0:
        return none
    if not (spec.flags & A.F_LOST_SALES) or not (spec.flags & A.F_CLAMP_INV):
        return none
    if spec.q_mul != 1.0 or spec.q_div != 1.0:
        return none
    if spec.deposit_rate != 0.0 or spec.overhead_rate != 0.0 or spec.penalty_cost != 0.0 or spec.hold_cost != 0.0:
        return none
    if not all(_small_int(x) for x in (spec.fixed_cost, spec.cash_min, spec.cash_max, spec.inv_min)) or spec.inv_min < 0:
        return none
    nI, nW = dims(spec)
    out = []
    for t in range(spec.T):
        price, v, ovh = (_per_period(spec, f, t) for f in ("price", "vari_cost", "overhead"))
        di = [int(d) for d in np.asarray(spec.pmf[t])[:, 0]]
        D = len(di)
        ok = _small_int(price, 32768) and _small_int(v, 32768) and _small_int(ovh) and v > 0
        ok = ok and all(di[j] == di[0] + j for j in range(D))
        if ok:
            big = (abs(price) * (abs(spec.inv_max) + spec.max_order_idx + abs(di[0]) + D) + abs(spec.cash_min) +
                   abs(spec.cash_max) + abs(v) * spec.max_order_idx + abs(spec.fixed_cost) + abs(ovh))
            ok = not (big > 5e8 or float(nI) * nW > 2.0e9)
        out.append((int(price), int(v), int(ovh), di[0]) if ok else None)
    return out


def cash_int_smem(D):
    return D * 28 + 16


def cash_diag_smem(D):
    return ((D * 24 + 15) & ~15) + 16


def cash_diag_ok(spec, plan, D):
    price, _, _, d0 = plan
    nI, nW = dims(spec)
    return (price > 0 and price * 7 <= nW and (nI + D + abs(d0) + 16 + spec.max_order_idx) * nW < 0x7fffffff and
            -(-nI // 8) <= 65535 and cash_diag_smem(D) <= 200 * 1024)


def cash_int_shape(spec, t, lo, hi):
    """-> (wide, parts) as cash_int_shape."""
    nI, nW = dims(spec)
    sms = sm_count()
    rows = (hi - 1) // nW - lo // nW + 1
    surv = spec.recursion == A.REC_SURVIVAL
    want = 64 * sms
    max_parts = max(1, min(16, (spec.max_order_idx + 1) // 12))

    def parts_for(tiles):
        return 1 if tiles >= want else min(-(-want // tiles), max_parts)
    tiles16 = rows * -(-nW // 1024)
    wide = t == spec.T and not surv and nW >= 512 and tiles16 * parts_for(tiles16) >= 2 * sms
    tile = 1024 if wide else 256
    parts = parts_for(rows * -(-nW // tile))
    if wide and tiles16 >= 3 * sms:
        parts = 1
    return wide, parts


def cash_diag_parts(spec, price, lo, hi):
    _, nW = dims(spec)
    ix0, ix1 = lo // nW, (hi - 1) // nW
    tiles = -(-(nW + price * 7) // 64) * -(-(ix1 - ix0 + 1) // 8)
    want = 256 * sm_count()
    parts = 1 if tiles >= want else min(-(-want // tiles), 16)
    return max(1, min(parts, (spec.max_order_idx + 1) // 12))


def _signbit_unit_cost(spec):
    return any(np.signbit(_per_period(spec, "vari_cost", t)) for t in range(spec.T))


def fallback(spec, D, request):
    """The row-shared or generic kernel a period takes when the integer kernels do not (plan_cash_tail, cash_row_ok)."""
    grows = not _signbit_unit_cost(spec)
    fits = D * 48 <= 96 * 1024
    if (request != ROW and spec.recursion == A.REC_EXPECT and fits and grows and 1.0 - spec.overhead_rate >= 0.0 and
            all(_per_period(spec, "price", t) >= 0.0 for t in range(spec.T)) and
            tail_bound(spec) * abs(spec.q_mul) < 2 ** 30 and spec.quantiser != A.Q_TRUNC):
        return TAIL
    return ROW if fits and grows else GENERIC


def predict(spec, request=AUTO, lo=0, hi=None):
    """-> ([(kernel, key, parts)] per period, launches, reported kernel) of a solve over [lo, hi), as
    choose_period_kernel and solve_period pick and count them."""
    nI, nW = dims(spec)
    hi = nI * nW if hi is None else hi
    plans = plan_cash(spec)
    surv = spec.recursion == A.REC_SURVIVAL
    is_min = not surv and spec.direction == MIN
    per = []
    for t in range(1, spec.T + 1):
        D, plan = len(spec.pmf[t - 1]), plans[t - 1]
        if request == GENERIC:
            per.append((GENERIC, None, 1))
        elif plan is not None and spec.terminal_value is None and hi > lo:
            if request != INT and t < spec.T and cash_diag_ok(spec, plan, D):
                parts = cash_diag_parts(spec, plan[0], lo, hi)
                per.append((DIAG, ("diag", surv, is_min, parts > 1), parts))
            elif cash_int_smem(D) <= 200 * 1024:
                wide, parts = cash_int_shape(spec, t, lo, hi)
                per.append((INT, ("int", surv, is_min, t == spec.T, 16 if wide else 4, parts > 1), parts))
            else:
                per.append((fallback(spec, D, request), None, 1))
        else:
            per.append((fallback(spec, D, request), None, 1))
    launches = sum(1 + (parts > 1) for _, _, parts in per)
    reported = 0
    for kernel, _, _ in reversed(per):   # periods T .. 1; GENERIC does not replace a specialised kernel, INT not DIAG
        if not (kernel == GENERIC and reported != 0) and not (kernel == INT and reported == DIAG):
            reported = kernel
    return per, launches, reported


ALL_KEYS = ({("diag", surv, mn, sl) for surv, mn in ((True, False), (False, True), (False, False)) for sl in (False, True)} |
            {("int", surv, mn, last, r, sl)
             for surv, mn, last, r in ((True, False, True, 4), (False, True, True, 4), (False, False, True, 4),
                                       (False, True, True, 16), (False, False, True, 16), (True, False, False, 4),
                                       (False, True, False, 4), (False, False, False, 4))
             for sl in (False, True)})


# ---- models and the check ---------------------------------------------------------------------------------------------
def cpmf(T, D, d0=0, seed=0, gap=None):
    """T rows of D consecutive integer demands from d0 (one point moved up by one when `gap` names a period)."""
    rng = np.random.default_rng(seed)
    rows = []
    for t in range(T):
        d = np.arange(d0, d0 + D, dtype=float)
        if gap == t:
            d[-1] += 1.0
        rows.append(np.stack([d, rng.dirichlet(np.ones(D))], axis=1))
    return rows


def int_model(pmf, price=3.0, v=1.0, K=2.0, ovh=1.0, inv=(0.0, 12.0), cash=(-10.0, 60.0), max_order=11, direction=MAX,
              gamma=1.0, surv=False, salvage=0.5, attrs=None, **kw):
    spec = S.cash_constraint_model(pmf, price=price, vari_cost=v, fixed_cost=K, salvage=salvage, overhead=ovh,
                                   max_order=max_order, inv_min=inv[0], inv_max=inv[1], cash_min=cash[0],
                                   cash_max=cash[1], quantiser=A.Q_LONGDIV, q_mul=1.0, q_div=1.0, gamma=gamma,
                                   direction=direction, recursion=A.REC_SURVIVAL if surv else A.REC_EXPECT, **kw)
    for k, val in (attrs or {}).items():
        setattr(spec, k, val)
    return spec


def _compare(tag, spec, request, st, t, V, Q, Vo, Qo):
    bad = np.flatnonzero((V.view(np.uint64) != Vo.view(np.uint64)) | (Q != Qo))
    assert len(bad) == 0, (f"{tag} request={request} ran {st['kernel_used']} t={t}: {len(bad)} states differ, first "
                           f"{bad[:3]} V {V[bad[:3]]} vs {Vo[bad[:3]]}, Q {Q[bad[:3]]} vs {Qo[bad[:3]]}")


def _check(spec, oracle, requests=(AUTO,), tag="", dense=None):
    """Whole grid, every period, bit for bit against the oracle for each request and the generic kernel; the reported
    kernel and the launch count must be the mirror's.  Returns the instantiation keys the requests reached."""
    Vo, Qo, evals, _ = dense if dense is not None else oracle.dense(spec)
    keys = set()
    for request in tuple(requests) + (GENERIC,):
        per, launches, reported = predict(spec, request)
        with S.Solver(spec, kernel=request) as s:
            s.solve()
            st = s.stats()
            for t in range(1, spec.T + 1):
                V, Q = s.period_tables(t)
                _compare(tag, spec, request, st, t, V, Q, Vo[t - 1], Qo[t - 1])
        assert st["evals"] == evals, (tag, request)
        assert st["kernel_used"] == reported, (tag, request, st["kernel_used"], reported, per)
        assert st["launches"] == launches, (tag, request, st["launches"], launches, per)
        keys |= {key for _, key, _ in per if key is not None}
    return keys


def _sample_check(oracle, spec, s, n=64, seed=3):
    """Period by period: V_t, Q_t at a seeded sample recomputed on the CPU from the solve's own V_{t+1}, bit for bit."""
    rng = np.random.default_rng(seed)
    idx = np.unique(np.concatenate([[0, s.n_states - 1], rng.integers(0, s.n_states, n)]))
    Vn = None
    for t in range(spec.T, 0, -1):
        V, Q = s.period_tables(t)
        vo, qo = oracle.step_states(spec, t, Vn, idx)
        assert np.array_equal(V[idx].view(np.uint64), vo.view(np.uint64)) and np.array_equal(Q[idx], qo), f"period {t}"
        Vn = V


def _check_large(spec, oracle, request, want_kernels, tag):
    """A grid too large for a whole-grid oracle: the solve against the generic kernel whole grid, and a seeded sample
    of every period against the oracle, inductively."""
    per, launches, reported = predict(spec, request)
    assert [k for k, _, _ in per] == list(want_kernels), (tag, per)
    with S.Solver(spec, kernel=request) as s, S.Solver(spec, kernel=GENERIC) as g:
        s.solve()
        g.solve()
        st = s.stats()
        assert st["kernel_used"] == reported and st["launches"] == launches, (tag, st["kernel_used"], st["launches"], per)
        assert st["evals"] == g.stats()["evals"]
        for t in range(1, spec.T + 1):
            V, Q = s.period_tables(t)
            Vg, Qg = g.period_tables(t)
            _compare(tag, spec, request, st, t, V, Q, Vg, Qg)
        _sample_check(oracle, spec, s)


# ---- a. every instantiation, sliced and unsliced ----------------------------------------------------------------------
def coverage_jobs():
    """(model, requests): two-period models reach bi_cash_diag (t = 1) and the narrow last-period bi_cash_int, or, on
    request, bi_cash_int with a successor; one-period models with >= 512 cash levels reach the wide last period."""
    jobs = []
    for surv in (False, True):
        for direction in ((MAX,) if surv else (MAX, MIN)):
            for mo in (11, 47):           # (mo + 1) / 12 = 1 or 4 slices at most
                jobs.append((int_model(cpmf(2, 6, 1, seed=mo), max_order=mo, direction=direction, surv=surv,
                                       cash=(-10.0, 60.0)), (AUTO, INT)))
    for direction in (MAX, MIN):
        # 25 rows x 1 tile of 1024: sliced 16 times; 450 rows: >= 3 tiles per SM, unsliced
        jobs.append((int_model(cpmf(1, 8, 0, seed=3), inv=(0.0, 24.0), cash=(-40.0, 559.0), max_order=191,
                               direction=direction), (AUTO,)))
        jobs.append((int_model(cpmf(1, 6, 0, seed=4), inv=(0.0, 449.0), cash=(-20.0, 499.0), max_order=5,
                               direction=direction), (AUTO,)))
    return jobs


def test_every_integer_cash_instantiation(oracle):
    assert len(ALL_KEYS) == 22
    keys = set()
    for spec, requests in coverage_jobs():
        keys |= _check(spec, oracle, requests, tag="coverage")
    assert keys == ALL_KEYS, f"{len(keys & ALL_KEYS)}/22 keys on {sm_count()} SMs, missing {sorted(ALL_KEYS - keys)}"


# ---- b. slices and first-wins -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_order", [11, 23, 24, 35, 47, 95, 191, 200])
def test_action_slices_and_ties(max_order, oracle):
    """Unit cost 3: the cash-limited action count differs between the 8 diagonal slots of a bi_cash_diag thread (cash
    steps of price 2) and between the R levels of a bi_cash_int thread (64 apart), so some slices hold no action of some
    states.  A salvage equal to the unit cost ties every order beyond the largest demand in period T, and gamma = 1 carries
    the ties into period 1: the first optimum must win across slice boundaries."""
    keys = set()
    for surv, direction in ((False, MAX), (False, MIN), (True, MAX)):
        spec = int_model(cpmf(2, 9, 2, seed=max_order), price=2.0, v=3.0, K=0.0, ovh=2.0, salvage=3.0,
                         inv=(0.0, 14.0), cash=(-30.0, 400.0), max_order=max_order, direction=direction, surv=surv)
        keys |= _check(spec, oracle, (AUTO, INT), tag=f"max_order={max_order} surv={surv} dir={direction}")
    slices = {k[-1] for k in keys}
    assert slices == ({False} if max_order < 23 else {True}), (max_order, keys)


# ---- c. geometry of bi_cash_diag's demand loop ------------------------------------------------------------------------
def diag_blocks(spec, t=1):
    """The kinds of step bi_cash_diag's main loop takes in period t (< T): per thread (8 diagonal states) and action,
    the 10-step blocks of the in-stock run -- 'lin_in' (one running offset, cash inside the axis), 'lin_hi' (one running
    offset, cash at or above the upper clamp), 'slow' (a clamp changes state inside the block) -- then 'mixed' (some
    slots stocked out) and 'tail' (every slot stocked out)."""
    price, v, ovh, d0 = plan_cash(spec)[t - 1]
    nI, nW = dims(spec)
    D, K, mo = len(spec.pmf[t - 1]), int(spec.fixed_cost), spec.max_order_idx
    kmin, res, surv = int(round(spec.cash_min)), _per_period(spec, "reserve", t - 1), spec.recursion == A.REC_SURVIVAL
    nW1, row_max, inv_min = nW - 1, (nI - 1) * nW, int(spec.inv_min)
    cols = np.arange(-(-(nW + 7 * price) // 64) * 64)
    seen = set()
    for ix0 in range(0, nI, 8):
        nAmax = np.zeros(len(cols), dtype=int)
        for k in range(8):
            iw = cols - price * k
            valid = (iw >= 0) & (iw < nW) & (ix0 + k < nI)
            with np.errstate(divide="ignore", invalid="ignore"):
                bound = np.fmax(0.0, ((kmin + iw - res) - spec.reserve2) / v)
            n = np.fmin(float(mo), bound).astype(int) + 1
            nAmax = np.maximum(nAmax, np.where(valid, n, 0))
        xv0 = inv_min + ix0
        for ai in range(int(nAmax.max())):
            c = cols[nAmax > ai]
            CI = (K if ai > 0 else 0) + v * ai + ovh
            L0 = ix0 + ai - d0
            jy0 = min(max(xv0 + ai - d0, 0), D)
            jy7 = min(max(xv0 + 7 + ai - d0, 0), D)
            ro_run = (L0 - 3) * nW
            c_run = c + price * (ix0 + ai) - CI - price * (L0 - 3)
            j = 0
            while j + 10 <= jy0:
                rows_in = ro_run - 9 * nW >= 0 and ro_run <= row_max
                cash_in = (c_run >= 0) & (c_run + 9 * price <= nW1)
                cash_hi = c_run >= nW1
                if rows_in and not surv:
                    if cash_in.any():
                        seen.add("lin_in")
                    if cash_hi.any():
                        seen.add("lin_hi")
                if not rows_in or surv or not (cash_in | cash_hi).all():
                    seen.add("slow")
                ro_run -= 10 * nW
                c_run = c_run + 10 * price
                j += 10
            if jy7 > max(jy0, 0) and jy0 < D:
                seen.add("mixed")
            if jy7 < D:
                seen.add("tail")
    return seen


def geometry_jobs():
    jobs = []
    # nI mod 8: every residue, with inv_min > 0 (in-stock successors clamp to row 0) on the odd ones
    for r in range(8):
        inv_min = 3.0 if r % 2 else 0.0
        jobs.append(int_model(cpmf(2, 11, 1, seed=r), inv=(inv_min, inv_min + 16 + r - 1), max_order=13 + r,
                              cash=(-20.0, 90.0), direction=MAX if r % 3 else MIN))
    # nW + 7 price around multiples of 64 (price 3 or 5)
    for price, span in ((3, 127), (3, 128), (3, 129), (5, 191), (5, 192), (5, 193)):
        nW = span - 7 * price
        jobs.append(int_model(cpmf(2, 12, 0, seed=span), price=float(price), inv=(0.0, 20.0), cash=(-15.0, nW - 16.0),
                              max_order=17))
    # demand tables shorter and longer than the 10-entry window, supports starting at 0, 1 and 5; stock above the
    # largest demand and at or below d0; large orders push y - d above inv_max
    for i, D in enumerate((1, 2, 7, 8, 9, 10, 11, 19, 20, 21)):
        d0 = (0, 1, 5)[i % 3]
        jobs.append(int_model(cpmf(2, D, d0, seed=100 + D), price=2.0, inv=(0.0, 9.0 + i), cash=(-25.0, 70.0),
                              max_order=26, direction=(MAX, MIN)[i % 2], gamma=(1.0, 0.9)[i % 2]))
    # cash bases below 0, inside, and at / above the upper clamp: a small axis and a wide price, a high reserve, and
    # the survival recursion (no running-offset blocks)
    jobs.append(int_model(cpmf(2, 25, 0, seed=7), price=4.0, v=1.0, inv=(0.0, 40.0), cash=(-5.0, 40.0), max_order=30))
    jobs.append(int_model(cpmf(2, 30, 2, seed=8), price=1.0, v=2.0, K=5.0, ovh=7.0, inv=(1.0, 45.0), cash=(-60.0, 30.0),
                          max_order=40, direction=MIN))
    jobs.append(int_model(cpmf(2, 22, 0, seed=9), price=3.0, inv=(0.0, 33.0), cash=(-10.0, 200.0), max_order=35,
                          surv=True))
    return jobs


def test_cash_diag_geometry(oracle):
    seen = set()
    for n, spec in enumerate(geometry_jobs()):
        assert predict(spec)[0][0][0] == DIAG, n
        _check(spec, oracle, (AUTO, INT), tag=f"geometry #{n}")
        seen |= diag_blocks(spec)
    assert seen == {"lin_in", "lin_hi", "slow", "mixed", "tail"}, seen


@pytest.mark.parametrize("nW", [255, 256, 257, 511, 512, 513, 1023, 1024, 1025])
def test_cash_int_geometry(nW, oracle):
    """bi_cash_int tiles of 256 (and 1024 in a wide last period) cash levels: the last tile full, one level short and
    one level over."""
    for direction in (MAX, MIN):
        spec = int_model(cpmf(2, 7, 1, seed=nW), inv=(0.0, 5.0), cash=(-30.0, nW - 31.0), max_order=25,
                         direction=direction)
        _check(spec, oracle, (AUTO, INT), tag=f"nW={nW}")
    # one period, many rows: the last period runs 16 levels per thread from 512 levels up
    spec = int_model(cpmf(1, 5, 0, seed=nW), inv=(0.0, 449.0), cash=(0.0, nW - 1.0), max_order=4)
    _check(spec, oracle, tag=f"nW={nW} T=1")


# ---- d. plan edges --------------------------------------------------------------------------------------------------
def _expect_kernels(spec, request, kernels, tag):
    got = [k for k, _, _ in predict(spec, request)[0]]
    assert got == list(kernels), (tag, got, kernels)


@pytest.mark.parametrize("price", [1, 3, 37])
def test_diagonal_fits_cash_axis_edge(price, oracle):
    """price * 7 <= nW: on the edge bi_cash_diag runs period 1, one level short bi_cash_int does."""
    for nW, first in ((7 * price, DIAG), (7 * price - 1, INT)):
        spec = int_model(cpmf(2, 6, 1, seed=nW), price=float(price), inv=(0.0, 11.0), cash=(-3.0, nW - 4.0), max_order=24)
        _expect_kernels(spec, AUTO, (first, INT), f"price {price} nW {nW}")
        _check(spec, oracle, tag=f"price {price} nW {nW}")


def test_price_zero_and_negative(oracle):
    for prices in ([0.0, 3.0], [-2.0, 3.0], [3.0, 0.0], [3.0, -1.0]):
        spec = int_model(cpmf(2, 6, 1, seed=5), attrs=dict(price_t=prices), max_order=30)
        _expect_kernels(spec, AUTO, (INT if prices[0] <= 0 else DIAG, INT), prices)
        _check(spec, oracle, (AUTO, INT), tag=f"price_t={prices}")


PERIOD_OUT = {   # period 2 of 3 leaves the plan; periods 1 and 3 stay in it
    "v_zero": dict(vari_cost_t=[1.0, 0.0, 2.0]),
    "v_minus_zero": dict(vari_cost_t=[1.0, -0.0, 2.0]),
    "v_negative": dict(vari_cost_t=[1.0, -1.0, 2.0]),
    "v_half": dict(vari_cost_t=[1.0, 0.5, 2.0]),
    "price_fraction": dict(price_t=[3.0, 4.5, 2.0]),
    "price_32767": dict(price_t=[3.0, 32767.0, 2.0]),
    "price_32768": dict(price_t=[3.0, 32768.0, 2.0]),
    "v_32767": dict(vari_cost_t=[1.0, 32767.0, 2.0]),
    "v_32768": dict(vari_cost_t=[1.0, 32768.0, 2.0]),
    "overhead_fraction": dict(overhead_t=[1.0, 2.5, 3.0], reserve_t=[1.0, 2.5, 3.0]),
    "demand_gap": "gap",
}


@pytest.mark.parametrize("case", list(PERIOD_OUT))
def test_one_period_leaves_the_plan(case, oracle):
    attrs = PERIOD_OUT[case]
    pmf = cpmf(3, 7, 1, seed=11, gap=1 if attrs == "gap" else None)
    for direction in (MAX, MIN):
        spec = int_model(pmf, cash=(-10.0, 80.0), max_order=29, direction=direction,
                         attrs=None if attrs == "gap" else attrs)
        plans = plan_cash(spec)
        inside = case.endswith("32767")
        assert plans[0] is not None and plans[2] is not None and (plans[1] is not None) == inside, (case, plans)
        _check(spec, oracle, (AUTO, INT), tag=case)


MODEL_OUT = {   # (attrs, integer kernels?)
    "hold": (dict(hold_cost=0.5), False), "hold_minus_zero": (dict(hold_cost=-0.0), True),
    "deposit": (dict(deposit_rate=0.25), False), "deposit_minus_zero": (dict(deposit_rate=-0.0), True),
    "overhead_rate": (dict(overhead_rate=0.125), False), "overhead_rate_minus_zero": (dict(overhead_rate=-0.0), True),
    "penalty": (dict(penalty_cost=0.5), False), "penalty_minus_zero": (dict(penalty_cost=-0.0), True),
    "fixed_fraction": (dict(fixed_cost=2.5, reserve2=2.5), False),
    "step_half": (dict(step=0.5), False),
    "q_2_2": (dict(q_mul=2.0, q_div=2.0), False),
    "q_div_1_1": (dict(quantiser=A.Q_DIV), True),
    "q_longdiv_1_1": (dict(quantiser=A.Q_LONGDIV), True),
}


@pytest.mark.parametrize("case", list(MODEL_OUT))
def test_model_wide_refusals(case, oracle):
    attrs, inside = MODEL_OUT[case]
    for direction in (MAX, MIN):
        spec = int_model(cpmf(2, 7, 1, seed=12), cash=(-10.0, 80.0), max_order=29, direction=direction, attrs=attrs)
        assert all((p is not None) == inside for p in plan_cash(spec)), case
        _check(spec, oracle, (AUTO, INT), tag=case)


def test_magnitude_guard_edge(oracle):
    """|price| * (|inv_max| + max_order + |d0| + D) + ... <= 5e8 with price 32767: inv_max on the last admitted value
    and one above."""
    def at(inv_max):
        return int_model(cpmf(2, 4, 1, seed=13), price=32767.0, inv=(0.0, float(inv_max)), cash=(-5.0, 4.0), max_order=3)

    def big(spec):   # plan_cash's terms in the same order
        D, d0 = len(spec.pmf[0]), int(spec.pmf[0][0, 0])
        return (abs(spec.price) * (abs(spec.inv_max) + spec.max_order_idx + abs(d0) + D) + abs(spec.cash_min) +
                abs(spec.cash_max) + abs(spec.vari_cost) * spec.max_order_idx + abs(spec.fixed_cost) + abs(spec.overhead))
    x = int((5e8 - big(at(0))) / 32767)
    while big(at(x)) > 5e8:
        x -= 1
    while big(at(x + 1)) <= 5e8:
        x += 1
    assert 14000 < x < 16000
    for inv_max, used in ((x, INT), (x + 1, TAIL)):
        spec = at(inv_max)
        _expect_kernels(spec, AUTO, (used, used), f"inv_max {inv_max}")
        _check(spec, oracle, (AUTO, INT), tag=f"inv_max {inv_max}")


def _long_pmf(T, D, seed):
    return cpmf(T, D, 0, seed=seed)


@pytest.mark.parametrize("D,kernels", [(1754, (INT,)), (1755, (INT,)), (7313, (INT,)), (7314, (GENERIC,))])
def test_cash_int_shared_memory_edge(D, kernels, oracle):
    """28 D + 16 bytes: 1754 points fit the default 48 KB, 1755 need the opt-in attribute, 7313 fit 200 KB."""
    spec = int_model(_long_pmf(1, D, D), inv=(0.0, 3.0), cash=(-3.0, 12.0), max_order=25)
    _expect_kernels(spec, AUTO, kernels, f"D={D}")
    _check(spec, oracle, tag=f"D={D}")


@pytest.mark.parametrize("D,first", [(2047, DIAG), (2048, DIAG), (8532, DIAG), (8533, GENERIC)])
def test_cash_diag_shared_memory_edge(D, first, oracle):
    """round16(24 D) + 16 bytes: 2047 points fit the default 48 KB, 2048 need the opt-in attribute, 8532 fit 200 KB;
    at 8533 neither integer kernel's tables fit."""
    spec = int_model(_long_pmf(2, D, D), price=1.0, inv=(0.0, 3.0), cash=(-3.0, 12.0), max_order=25)
    _expect_kernels(spec, AUTO, (first, INT if D < 7314 else GENERIC), f"D={D}")
    _check(spec, oracle, tag=f"D={D}")


def test_shared_memory_edges_inside_one_model(oracle):
    rng = np.random.default_rng(17)
    pmf = [np.stack([np.arange(D, dtype=float), rng.dirichlet(np.ones(D))], axis=1) for D in (8533, 8532, 7314, 7313)]
    spec = int_model(pmf, price=1.0, inv=(0.0, 2.0), cash=(-3.0, 10.0), max_order=13)
    _expect_kernels(spec, AUTO, (GENERIC, DIAG, DIAG, INT), "mixed D")
    _expect_kernels(spec, INT, (GENERIC, GENERIC, GENERIC, INT), "mixed D")
    _check(spec, oracle, (AUTO, INT), tag="mixed D")


def test_cash_diag_row_offset_edge(oracle):
    """(nI + D + |d0| + 16 + max_order) * nW < 2^31 - 1: with 2^21 - 1 cash levels and one inventory row the sum is
    1024 (bi_cash_diag) or 1025 (bi_cash_int)."""
    for D, first in ((1004, DIAG), (1005, INT)):
        spec = int_model(_long_pmf(2, D, 21), price=5.0, v=40000.0 / 4, K=0.0, ovh=3.0, inv=(0.0, 0.0),
                         cash=(-1048575.0, 1048575.0), max_order=3)
        nI, nW = dims(spec)
        assert (nI + D + 16 + 3) * nW - 0x7fffffff == (-1023 if D == 1004 else 2096128)
        _check_large(spec, oracle, AUTO, (first, INT), f"D={D}")


def test_cash_diag_grid_y_limit(oracle):
    """bi_cash_diag puts ceil(rows / 8) tiles on gridDim.y: 524,280 inventory rows are 65535 tiles, 524,281 one more,
    which the plan must refuse (the period runs bi_cash_int) rather than fail the launch."""
    for rows, first in ((524280, DIAG), (524281, INT)):
        spec = int_model(cpmf(2, 3, 0, seed=19), price=1.0, inv=(0.0, rows - 1.0), cash=(0.0, 9.0), max_order=3)
        _check_large(spec, oracle, AUTO, (first, INT), f"rows={rows}")


def test_cash_int_widest_cash_axis(oracle):
    """plan_cash keeps |cash_min|, |cash_max| < 2^20, so bi_cash_int's gridDim.y (ceil(nW / 256) cash tiles) is at most
    8192: the widest admitted axis runs it, one level more is refused."""
    for cash_max, used in ((1048575.0, INT), (1048576.0, ROW)):
        spec = int_model(cpmf(1, 3, 0, seed=23), inv=(0.0, 0.0), cash=(-1048575.0, cash_max), max_order=3, surv=True)
        _expect_kernels(spec, AUTO, (used,), f"cash_max {cash_max}")
        _check(spec, oracle, tag=f"cash_max {cash_max}")


# ---- e. survival ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cash", [(-40.0, 150.0), (0.0, 150.0), (5.0, 150.0)])
def test_survival(cash, oracle):
    """Successors with negative cash read 0 (cash_min < 0); none exist for cash_min >= 0.  Last-period scoring sliced
    and unsliced."""
    for mo in (11, 47):
        spec = int_model(cpmf(3, 8, 1, seed=mo), price=4.0, v=2.0, K=1.0, ovh=6.0, inv=(0.0, 17.0), cash=cash,
                         max_order=mo, surv=True, attrs=dict(price_t=[4.0, 5.0, 3.0], overhead_t=[6.0, 9.0, 4.0]))
        _check(spec, oracle, (AUTO, INT), tag=f"survival cash={cash} mo={mo}")


# ---- f. shards ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3, 5, 8])
def test_shards_sliced(world, oracle):
    """Sliced launches on every shard, so merge_action_slices stores the merged rows into the peers' tables; shard
    edges cut through 8-row tiles and through rows; with 7 states in 8 shards one shard is empty."""
    jobs = [int_model(cpmf(2, 9, 1, seed=world), inv=(0.0, 19.0), cash=(-13.0, 40.0), max_order=47),
            int_model(cpmf(2, 6, 0, seed=world), inv=(0.0, 12.0), cash=(-20.0, 30.0), max_order=95, direction=MIN),
            int_model(cpmf(2, 7, 2, seed=world), inv=(0.0, 9.0), cash=(-10.0, 60.0), max_order=35, surv=True)]
    if world == 8:
        jobs.append(int_model(cpmf(2, 4, 0, seed=8), price=1.0, inv=(0.0, 0.0), cash=(0.0, 6.0), max_order=47))
    for spec in jobs:
        Vo, Qo, evals, _ = oracle.dense(spec)
        for request in (AUTO, INT):
            with S.Group(spec, [0] * world, kernel=request) as g:
                g.solve()
                for t in range(1, spec.T + 1):
                    V, Q = g.period_tables(t)
                    assert np.array_equal(V.view(np.uint64), Vo[t - 1].view(np.uint64)) and np.array_equal(Q, Qo[t - 1]), \
                        (spec.name, world, request, t)
                assert g.stats()["evals"] == evals
                ran = 0
                for sh in g.shards:
                    lo, hi = sh.grid.shard_lo, sh.grid.shard_hi
                    if hi <= lo:
                        continue
                    ran += 1
                    per, _, reported = predict(spec, request, lo, hi)
                    assert sh.stats()["kernel_used"] == reported, (world, request, lo, hi, per)
                    assert reported == (DIAG if request == AUTO else INT), (world, request, per)
                    assert any(parts > 1 for _, _, parts in per), (world, request, lo, hi, per)
                assert ran == min(world, g.n_states)


# ---- g. seeded fuzz -------------------------------------------------------------------------------------------------
def fuzz_model(rng, surv):
    while True:
        T = int(rng.integers(1, 5))
        D = int(rng.integers(1, 301)) if rng.random() < 0.5 else int(rng.integers(1, 21))
        d0 = int(rng.integers(0, 6))
        pmf = cpmf(T, D, d0, seed=int(rng.integers(1 << 30)),
                   gap=int(rng.integers(T)) if rng.random() < 0.1 and D > 1 else None)
        mo = int(rng.choice([int(rng.integers(0, 24)), int(rng.integers(24, 201))]))
        inv_min = float(rng.integers(0, 4))
        inv_max = inv_min + float(rng.integers(0, 40))
        nW = int(rng.integers(1, 1501))
        cash_min = float(rng.integers(-nW, 1)) if rng.random() < 0.8 else float(rng.integers(0, 30))
        kw = dict(price=float(rng.integers(-1, 12)), v=float(rng.integers(1, 6)), K=float(rng.integers(-3, 6)),
                  ovh=float(rng.integers(-4, 8)), salvage=float(rng.choice([0.0, 0.5, 1.0, 2.0])),
                  inv=(inv_min, inv_max), cash=(cash_min, cash_min + nW - 1), max_order=mo,
                  gamma=float(rng.choice([1.0, 0.9])), direction=MAX if surv else int(rng.choice([MAX, MIN])), surv=surv)
        attrs = {}
        if rng.random() < 0.5:
            attrs["price_t"] = [float(rng.integers(0, 12)) for _ in range(T)]
            attrs["vari_cost_t"] = [float(rng.integers(1, 6)) for _ in range(T)]
            attrs["overhead_t"] = [float(rng.integers(-4, 8)) for _ in range(T)]
            attrs["reserve_t"] = list(attrs["overhead_t"])
            if rng.random() < 0.3:   # one period out of the plan
                t = int(rng.integers(T))
                key, val = [("price_t", 4.5), ("vari_cost_t", 0.5), ("vari_cost_t", 0.0), ("overhead_t", 1.5)][int(rng.integers(4))]
                attrs[key][t] = val
        spec = int_model(pmf, attrs=attrs, **kw)
        nI, nW = dims(spec)
        if nI * nW * (mo + 1) * sum(len(r) for r in pmf) <= 2e8:
            return spec


@pytest.mark.parametrize("family", ["expect", "survival"])
def test_fuzz_integer_cash(family, oracle):
    rng = np.random.default_rng(4242 + (family == "survival"))
    iters = int(os.environ.get("SDPB_FUZZ_ITERS", "40"))   # raise for a longer one-off campaign
    integer = 0
    for it in range(iters):
        spec = fuzz_model(rng, family == "survival")
        _check(spec, oracle, (AUTO, INT), tag=f"{family} #{it}")
        integer += any(k in (DIAG, INT) for k, _, _ in predict(spec)[0])
    assert integer >= iters // 2, f"only {integer} of {iters} models ran an integer kernel"
