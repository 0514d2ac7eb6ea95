"""The reached-state engine kept as a handle (sdpb_reached_*): every reached state queryable, extension with states of
any period, and the policy rolled out over sample paths, for all four kinds (CashRecursionMultiLead,
CashRecursionMultiXR, CashRecursionV, CashRecursionRounded).

Every GPU comparison is bit for bit (==) against the oracle's literal memoised recursions (tests/reached_oracle.py):
reached_at for the same getExpectedValue calls, reached_simulate for the same roll-out."""
from __future__ import annotations

import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

import reached_oracle as RO
from test_parity_gpu import _multi_pmf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp = C.POINTER(C.c_double)


def _arr(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


# ---- small instances of every kind: (facade, root, state class) --------------------------------------------------------
def _multilead(S, T=3, qb=7, ovh=100.0, vals=((10, 30), (5, 15)), probs=((0.5, 0.5), (0.5, 0.5))):
    """Cash goes below zero from the first period on (overhead 100, no initial cash): exercises the cash order."""
    rec = S.CashRecursionMultiLead(_multi_pmf(vals[0], probs[0], vals[1], probs[1], T), Qbound=qb, overheadCost=[ovh] * T)
    return rec, [0.0, 0.0, 0.0, 0.0, 0.0]


def _xr(S, T=2, qb=8, cash=25.0, pmf=None):
    pmf = pmf or S.GetPmfMulti([[S.PoissonDist(4)] * T, [S.PoissonDist(3)] * T], 0.99, 1).tables()
    rec = S.CashRecursionMultiXR(pmf, price=(5, 10), variCost=(1, 2), Qbound=qb, maxInventoryState=40, maxCashState=500)
    return rec, [0.0, 0.0, cash]


def _yr(S, T=2, qb=8, cash=10.0, dr=0.0):
    pmf = S.GetPmfMulti([[S.PoissonDist(4)] * T, [S.PoissonDist(3)] * T], 0.99, 1).tables()
    rec = S.CashRecursionV(pmf, price=(5, 10), variCost=(1, 2), depositeRate=dr, Qbound=qb, maxInventoryState=40,
                           maxCashState=500)
    return rec, [0.0, 0.0, cash]


def _rounded(S, means=(6, 3, 2, 5), K=8.0, cash=33.0, rate=0.0, maxQ=60):
    pmf = S.GetPmf([S.PoissonDist(m) for m in means], 0.9999, 1).getpmf()
    rec = S.CashRecursionRounded(pmf, price=4, variCost=1, fixOrderCost=K, holdingCost=0, salvageValue=0.5,
                                 interestRate=rate, minCashRequired=0, maxOrderQuantity=maxQ, maxInventoryState=500,
                                 minCashState=-100, maxCashState=2000)
    return rec, [0.0, cash]


KINDS = {"multilead": _multilead, "xr": _xr, "yr": _yr, "rounded": _rounded}


def _pmf_rows(rec):
    """per period: (demand rows [D, nd], probabilities [D]) as the engine holds them"""
    T, nD = rec.T, rec._m.n_demands
    d1, d2, p = rec._d1.reshape(T, nD), rec._d2.reshape(T, nD), rec._p.reshape(T, nD)
    out = []
    for t in range(T):
        n = rec._lens[t]
        d = np.column_stack([d1[t, :n], d2[t, :n]]) if rec.kind != 3 else d1[t, :n, None]
        out.append((d, p[t, :n]))
    return out


def _snapshot(rh):
    st = rh.stats()
    return rh.opt_table(), rh.n_states(), st["evals"], st["evals_executed"]


def _assert_memo(rh, rows, ev, what):
    """opt_table, the value and action of every reached state, and evals == the oracle's memo [t, state..., a1, a2, V]"""
    nd = rh.ndim
    tab = rh.opt_table()
    assert tab.shape == (len(rows), nd + 3), (what, tab.shape, rows.shape)
    assert np.array_equal(tab, rows[:, :-1]), what
    st = rh.stats()
    assert st["evals"] == ev and st["evals_executed"] == ev, (what, st["evals"], ev)
    assert sum(rh.n_states()) == len(rows), what
    for t in range(1, rh.T + 1):
        sel = rows[rows[:, 0] == t]
        if len(sel):
            v, a1, a2 = rh.value(t, sel[:, 1:1 + nd])
            assert np.array_equal(v, sel[:, -1]) and np.array_equal(a1, sel[:, -3]) and np.array_equal(a2, sel[:, -2]), \
                (what, t)


# ---- no GPU needed ----------------------------------------------------------------------------------------------------
def test_null_handle_is_an_argument_error(S):
    lib = S.abi.load()
    A = S.abi
    st, out = _arr([0.0] * 5), np.empty(4)
    n = C.c_size_t(0)
    ns = (C.c_int64 * 4)()
    stats = A.SdpbStats()
    assert lib.sdpb_reached_value(None, 1, st.ctypes.data_as(_dp), 1, None, None, None) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_extend(None, 1, st.ctypes.data_as(_dp), 1) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_opt_table(None, None, C.byref(n)) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_states(None, ns) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_stats(None, C.byref(stats)) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_simulate(None, st.ctypes.data_as(_dp), out.ctypes.data_as(_dp), 1, 1.0,
                                     out.ctypes.data_as(_dp)) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_last_error()
    lib.sdpb_reached_destroy(None)


def test_open_argument_errors_and_no_device(S):
    import torch
    A = S.abi
    lib = A.load()
    rec, root = _multilead(S, T=2, qb=3)
    st = _arr(root)
    h = C.c_void_p()
    assert lib.sdpb_reached_open(None, -1, 0, st.ctypes.data_as(_dp), 1, C.byref(h)) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_open(C.byref(rec._m), -1, 0, st.ctypes.data_as(_dp), -1, C.byref(h)) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_open(C.byref(rec._m), -1, -1, st.ctypes.data_as(_dp), 1, C.byref(h)) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_open(C.byref(rec._m), -1, 0, None, 1, C.byref(h)) == A.SDPB_ERR_ARG
    rc = lib.sdpb_reached_open(C.byref(rec._m), -1, 0, st.ctypes.data_as(_dp), 1, C.byref(h))
    if torch.cuda.is_available():
        assert rc == A.SDPB_OK
        lib.sdpb_reached_destroy(h)
    else:
        assert rc == A.SDPB_ERR_NO_DEVICE and h.value is None
        assert b"device" in lib.sdpb_reached_last_error()


def test_cpp_reached_compiles(tmp_path):
    src = tmp_path / "reached.cpp"
    src.write_text('''#include "sdpb200.hpp"
using namespace sdpb200;
int main() {
    // CashRecursionMultiLead, T = 2, demands {10, 30} x {5, 15}, Qbound 6
    const int T = 2, nD = 4;
    std::vector<double> d1, d2, p, ovh(T, 100.0);
    for (int t = 0; t < T; t++)
        for (double a : {10.0, 30.0})
            for (double b : {5.0, 15.0}) { d1.push_back(a); d2.push_back(b); p.push_back(0.25); }
    sdpb_reached_model m;
    std::memset(&m, 0, sizeof m);
    m.struct_size = (uint32_t)sizeof m;
    m.kind = SDPB_REACHED_MULTILEAD; m.T = T; m.q_bound = 6; m.n_demands = nD;
    m.d1 = d1.data(); m.d2 = d2.data(); m.p = p.data(); m.overhead_t = ovh.data();
    m.price[0] = 5; m.price[1] = 10; m.vari_cost[0] = 1; m.vari_cost[1] = 2; m.salvage[0] = 0.5; m.salvage[1] = 1;
    m.r1 = 0.1; m.r2 = 2; m.limit = 500; m.max_inv = 200; m.min_cash = -500; m.max_cash = 5000;
    m.gamma = 1; m.tie_tolerance = 0.1;
    try {
        Reached r(m, {{0, 0, 0, 0, 0}});
        const std::array<double, 3> root = r.valueAndAction(1, {0, 0, 0, 0, 0});
        const sdpb_stats s0 = r.stats();
        r.extend(2, {{3, 1, 2, 2, -17.123}});
        const std::vector<double> v = r.simulate({0, 0, 0, 0, 0}, {{10, 5, 30, 15}, {31.4, 4.6, 9.5, 15}}, 1.0);
        const bool ok = v.size() == 2 && r.optTable().size() == r.nStates(1) + r.nStates(2) && r.stats().evals > s0.evals &&
                        root[0] == r.value(1, {0, 0, 0, 0, 0});
        return ok ? 0 : 1;
    } catch (const SdpbError& e) {
        return e.code == SDPB_ERR_NO_DEVICE ? 3 : 2;
    }
}
''')
    exe = tmp_path / "reached"
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                    "-o", str(exe), "-L", os.path.join(ROOT, "stochastic-inventory_b200"), "-lsdpb200",
                    "-Wl,-rpath," + os.path.join(ROOT, "stochastic-inventory_b200")], check=True)
    import torch
    rc = subprocess.run([str(exe)]).returncode
    assert rc == (0 if torch.cuda.is_available() else 3)


# ---- GPU: one-root open == sdpb_reached_solve ---------------------------------------------------------------------------
SOLVE_CASES = ([("multilead", dict(T=T, qb=qb, ovh=ovh)) for T, qb, ovh in [(3, 7, 100.0), (3, 9, 20.0), (4, 4, 35.0),
                                                                            (1, 12, 100.0)]]
               + [("multilead", dict(T=2, qb=50, vals=((20, 30, 40), (10, 15, 20)),
                                     probs=((0.25, 0.5, 0.25), (0.25, 0.5, 0.25))))]
               + [("xr", dict(T=T, qb=qb, cash=c)) for T, qb, c in [(2, 8, 0.0), (2, 12, 25.0), (3, 5, 10.0), (1, 10, 30.0)]]
               + [("yr", dict(T=T, qb=qb, cash=c, dr=dr)) for T, qb, c, dr in [(2, 8, 10.0, 0.0), (2, 12, 25.0, 0.05),
                                                                              (3, 5, 14.0, 0.0), (1, 10, 30.0, 0.0)]]
               + [("rounded", dict(means=m, K=K, cash=c, rate=r)) for m, K, c, r in [((6, 3, 2, 5), 8.0, 33.0, 0.0),
                                                                                     ((20, 7, 2, 14), 24.0, 33.0, 0.0),
                                                                                     ((5, 4, 6), 0.0, 27.0, 0.1)]])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,kw", SOLVE_CASES, ids=[f"{k}-{i}" for i, (k, _) in enumerate(SOLVE_CASES)])
def test_open_equals_reached_solve(kind, kw, S):
    rec, root = KINDS[kind](S, **kw)
    lib = S.abi.load()
    st = _arr(root)
    v, a1, a2, ms = C.c_double(), C.c_double(), C.c_double(), C.c_double()
    ns = (C.c_int64 * rec.T)()
    assert lib.sdpb_reached_solve(C.byref(rec._m), -1, st.ctypes.data_as(_dp), C.byref(v), C.byref(a1), C.byref(a2), ns,
                                  C.byref(ms)) == S.abi.SDPB_OK
    with S.Reached(rec._m, [root]) as rh:
        hv, h1, h2 = rh.value(1, [root])
        assert (hv[0], h1[0], h2[0]) == (v.value, a1.value, a2.value)
        assert rh.n_states() == list(ns)
        assert ms.value > 0 and rh.stats()["solve_ms"] > 0


# ---- GPU: the whole memo, extension, failures ----------------------------------------------------------------------------
MEMO_CASES = [("multilead", dict(T=3, qb=7, ovh=100.0)), ("multilead", dict(T=3, qb=9, ovh=20.0)),
              ("xr", dict(T=3, qb=5, cash=10.0)), ("yr", dict(T=3, qb=5, cash=14.0)),
              ("yr", dict(T=2, qb=8, cash=25.0, dr=0.05)), ("rounded", dict()),
              ("rounded", dict(means=(5, 4, 6), K=0.0, cash=27.0, rate=0.1, maxQ=20))]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,kw", MEMO_CASES, ids=[f"{k}-{i}" for i, (k, _) in enumerate(MEMO_CASES)])
def test_whole_memo_matches_oracle(kind, kw, S):
    rec, root = KINDS[kind](S, **kw)
    rows, vals, ev = RO.reached_at(rec._m, [1], [root])
    with S.Reached(rec._m, [root]) as rh:
        _assert_memo(rh, rows, ev, kind)
        assert rh.value(1, [root])[0][0] == vals[0]
    if kw.get("ovh") == 20.0:
        assert (rows[:, 5] < 0).any() and (rows[:, 5] > 0).any()  # both signs of cash in one period's order


def _unreached(rows, nd, t, k=3):
    """Up to k states of period t that no root reaches: reached ones with a fractional cash"""
    sel = rows[rows[:, 0] == t, 1:1 + nd][:k].copy()
    sel[:, -1] += 0.37
    return sel


@pytest.mark.gpu
@pytest.mark.parametrize("kind,kw", MEMO_CASES, ids=[f"{k}-{i}" for i, (k, _) in enumerate(MEMO_CASES)])
def test_extension_matches_oracle(kind, kw, S):
    """roots added one at a time, reached states of periods 2..T (no-op), unreached ones, then another root: after each
    step the handle == the oracle after the same getExpectedValue calls in the same order"""
    rec, root = KINDS[kind](S, **kw)
    nd = len(root)
    root2 = list(root)
    root2[-1] += 3.5
    calls = [(1, root)]
    rh = S.Reached(rec._m, [])
    rh.extend(1, [root])
    rows, _, ev = RO.reached_at(rec._m, *zip(*calls))
    _assert_memo(rh, rows, ev, (kind, "root"))
    before = _snapshot(rh)
    for t in range(2, rec.T + 1):
        sel = rows[rows[:, 0] == t, 1:1 + nd][:4]
        rh.extend(t, sel)
        calls += [(t, list(r)) for r in sel]
    after = _snapshot(rh)
    assert np.array_equal(after[0], before[0]) and after[1:] == before[1:]
    for t in range(2, rec.T + 1):
        new = _unreached(rows, nd, t)
        rh.extend(t, new)
        calls += [(t, list(r)) for r in new]
    want, _, ev = RO.reached_at(rec._m, *zip(*calls))
    assert len(want) > len(rows) or rec.T == 1
    _assert_memo(rh, want, ev, (kind, "later periods"))
    rh.extend(1, [root2])
    calls.append((1, root2))
    want, vals, ev = RO.reached_at(rec._m, *zip(*calls))
    _assert_memo(rh, want, ev, (kind, "second root"))
    assert rh.value(1, [root2])[0][0] == vals[-1]
    # one handle from both roots == the two roots one at a time (no later-period calls in between)
    both, _, ev2 = RO.reached_at(rec._m, [1, 1], [root, root2])
    with S.Reached(rec._m, [root, root2]) as rb:
        _assert_memo(rb, both, ev2, (kind, "two roots"))


@pytest.mark.gpu
def test_failed_extension_leaves_the_handle_as_it_was(S):
    A = S.abi
    rec, root = _multilead(S, T=3, qb=7)
    rows, _, _ = RO.reached_at(rec._m, [1], [root])
    s2 = rows[rows[:, 0] == 2, 1:6][:1]
    s3 = rows[rows[:, 0] == 3, 1:6][:1]
    # period 2 has one candidate, its 7 * 7 * 4 successors in period 3 need 196 * 16 * 2.2 bytes > 5000
    rh = S.Reached(rec._m, [], scratch_bytes=5000)
    rh.extend(3, s3)
    before = _snapshot(rh)
    with pytest.raises(S.SdpbError) as e:
        rh.extend(2, s2)
    assert e.value.code == A.SDPB_ERR_NOMEM and "period 3" in str(e.value), str(e.value)
    after = _snapshot(rh)
    assert np.array_equal(after[0], before[0]) and after[1:] == before[1:]
    want, _, ev = RO.reached_at(rec._m, [3], s3)
    _assert_memo(rh, want, ev, "after NOMEM")
    # an invalid root
    rh = S.Reached(rec._m, [root])
    before = _snapshot(rh)
    for bad in ([0.5, 0, 0, 0, 0.0], [0, 0, 70000, 0, 0.0], [-1, 0, 0, 0, 0.0]):
        with pytest.raises(S.SdpbError) as e:
            rh.extend(2, [root, bad])
        assert e.value.code == A.SDPB_ERR_OFFGRID
    with pytest.raises(S.SdpbError) as e:
        rh.simulate([0.5, 0, 0, 0, 0.0], np.ones((2, 3, 2)))
    assert e.value.code == A.SDPB_ERR_OFFGRID
    after = _snapshot(rh)
    assert np.array_equal(after[0], before[0]) and after[1:] == before[1:]
    # a state that has no key is simply not reached
    with pytest.raises(S.SdpbError) as e:
        rh.value(2, [[0.5, 0, 0, 0, 0.0]])
    assert e.value.code == A.SDPB_ERR_UNSOLVED
    rr, rroot = _rounded(S)
    with S.Reached(rr._m, [rroot]) as r3:
        with pytest.raises(S.SdpbError) as e:
            r3.extend(2, [[0.05, 10.0]])  # not k / 0.1
        assert e.value.code == A.SDPB_ERR_OFFGRID


@pytest.mark.gpu
def test_argument_errors(S):
    A = S.abi
    lib = A.load()
    rec, root = _yr(S)
    rh = S.Reached(rec._m, [root])
    before = _snapshot(rh)
    st = _arr([root])
    v = np.empty(1)
    for period, n in ((0, 1), (rec.T + 1, 1), (1, -1)):
        assert lib.sdpb_reached_extend(rh.h, period, st.ctypes.data_as(_dp), n) == A.SDPB_ERR_ARG
        assert lib.sdpb_reached_value(rh.h, period, st.ctypes.data_as(_dp), n, v.ctypes.data_as(_dp), None,
                                      None) == A.SDPB_ERR_ARG
    assert lib.sdpb_reached_extend(rh.h, 2, st.ctypes.data_as(_dp), 0) == A.SDPB_OK
    for bad in (np.nan, np.inf):
        for call in (lambda s: rh.extend(2, s), lambda s: rh.value(2, s)):
            with pytest.raises(S.SdpbError) as e:
                call([[0.0, 0.0, bad]])
            assert e.value.code == A.SDPB_ERR_ARG
    sm = np.ones((4, rec.T, 2))
    out = np.empty(4)
    sim = lib.sdpb_reached_simulate
    assert sim(rh.h, None, _arr(sm).ctypes.data_as(_dp), 4, 1.0, out.ctypes.data_as(_dp)) == A.SDPB_ERR_ARG
    assert sim(rh.h, st.ctypes.data_as(_dp), None, 4, 1.0, out.ctypes.data_as(_dp)) == A.SDPB_ERR_ARG
    assert sim(rh.h, st.ctypes.data_as(_dp), _arr(sm).ctypes.data_as(_dp), 0, 1.0, out.ctypes.data_as(_dp)) == A.SDPB_ERR_ARG
    with pytest.raises(S.SdpbError) as e:  # the V / Pi form has no per-period value to discount
        rh.simulate(root, sm, 0.9)
    assert e.value.code == A.SDPB_ERR_ARG
    nan_sm = sm.copy()
    nan_sm[1, 0, 1] = np.nan
    with pytest.raises(S.SdpbError) as e:
        rh.simulate(root, nan_sm)
    assert e.value.code == A.SDPB_ERR_ARG
    with pytest.raises(ValueError):
        rh.simulate(root, np.ones((4, rec.T, 1)))
    after = _snapshot(rh)
    assert np.array_equal(after[0], before[0]) and after[1:] == before[1:]


# ---- GPU: roll-out ----------------------------------------------------------------------------------------------------
def _support_samples(rec, n, seed):
    """demand draws from each period's pmf support (the exact demand values)"""
    rng = np.random.default_rng(seed)
    out = []
    for d, p in _pmf_rows(rec):
        out.append(d[rng.integers(0, len(d), size=n)])
    return np.stack(out, axis=1)  # [n, T, nd]


def _wild_samples(rec, n, seed):
    """fractional and out-of-support draws around the support (negative demands reach states no support draw does)"""
    rng = np.random.default_rng(seed)
    hi = max(float(d.max()) for d, _ in _pmf_rows(rec))
    nd = 1 if rec.kind == 3 else 2
    return rng.uniform(-4.4, hi + 6.0, size=(n, rec.T, nd))


ROLL_CASES = MEMO_CASES + [("multilead", dict(T=2, qb=12, ovh=100.0, vals=((20, 30, 40), (10, 15, 20)),
                                              probs=((0.25, 0.5, 0.25), (0.25, 0.5, 0.25))))]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,kw", ROLL_CASES, ids=[f"{k}-{i}" for i, (k, _) in enumerate(ROLL_CASES)])
def test_rollout_matches_oracle(kind, kw, S):
    rec, root = KINDS[kind](S, **kw)
    discounts = (1.0,) if kind == "yr" else (1.0, 0.9)
    grew = False
    for discount in discounts:
        for wild, samples in ((False, _support_samples(rec, 400, 3)), (True, _wild_samples(rec, 400, 4))):
            rh = S.Reached(rec._m, [root])
            n0 = rh.n_states()
            got = rh.simulate(root, samples, discount)
            want, rows, ev = RO.reached_simulate(rec._m, root, samples, discount)
            assert np.array_equal(got, want), (kind, wild, discount)
            _assert_memo(rh, rows, ev, (kind, wild, discount))
            rounds = rh.stats()["launches"]
            assert 1 <= rounds <= rec.T
            if not wild:
                assert rounds == 1 and rh.n_states() == n0  # every state a path meets was reached from the root
            grew |= rh.n_states() != n0
    assert grew or rec.T == 1


def _exhaustive(rec, root, rh):
    """every demand sequence with its probability: sum_paths w * value -> compare with V(root)"""
    rows = _pmf_rows(rec)
    paths, weights = [], []
    for combo in itertools.product(*[range(len(p)) for _, p in rows]):
        paths.append(np.stack([rows[t][0][j] for t, j in enumerate(combo)]))
        weights.append(np.prod([rows[t][1][j] for t, j in enumerate(combo)]))
    vals = rh.simulate(root, np.stack(paths), 1.0)
    return float(np.dot(np.asarray(weights), vals)), rh.value(1, [root])[0][0], len(paths)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,kw", [("multilead", dict(T=3, qb=7)),
                                     ("xr", dict(T=2, qb=6, pmf=_multi_pmf([2, 5], [0.5, 0.5], [1, 4], [0.25, 0.75], 2))),
                                     ("yr", dict(T=2, qb=6)),
                                     ("rounded", dict(means=(3, 2, 4), K=4.0, cash=20.0, maxQ=15))],
                         ids=["multilead", "xr", "yr", "rounded"])
def test_rollout_expectation_is_the_value(kind, kw, S):
    """(the pmf of each period sums to 1 where the value adds an immediate value per period: xr, multilead, rounded)"""
    rec, root = KINDS[kind](S, **kw)
    with S.Reached(rec._m, [root]) as rh:
        mean, v, n = _exhaustive(rec, root, rh)
    assert abs(mean - v) <= 1e-12 * abs(v), (kind, mean, v, n)


@pytest.mark.gpu
@pytest.mark.parametrize("vals,probs,value,n_paths",
                         [(((10, 30), (5, 15)), ((0.5, 0.5), (0.5, 0.5)), -76.56, 64),
                          (((20, 30, 40), (10, 15, 20)), ((0.25, 0.5, 0.25), (0.25, 0.5, 0.25)), 91.19499999999998, 729)],
                         ids=["T3-4pairs", "T3-9pairs"])
def test_rollout_expectation_on_the_recorded_instances(vals, probs, value, n_paths, S):
    """src/cash/overdraft/MultiProductLeadtime.java:35-39,45-50: the two recorded T = 3 outputs, 1.7e7 states each"""
    rec = S.CashRecursionMultiLead(_multi_pmf(vals[0], probs[0], vals[1], probs[1], 3), Qbound=50)
    root = [0.0] * 5
    with S.Reached(rec._m, [root]) as rh:
        mean, v, n = _exhaustive(rec, root, rh)
        assert v == value and n == n_paths
        assert rh.stats()["launches"] == 1
    assert abs(mean - v) <= 1e-12 * abs(v), (mean, v)


# ---- GPU: the facades ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_multilead_facade_answers_every_reached_state(S):
    """the recorded T = 2 instance (MultiProductLeadtime.java:41-43): getAction at period-2 states == the oracle memo, and
    getExpectedValue on a later-period state that was not reached extends the memo"""
    rec = S.CashRecursionMultiLead(_multi_pmf([20, 30, 40], [0.25, 0.5, 0.25], [10, 15, 20], [0.25, 0.5, 0.25], 2),
                                   Qbound=50)
    ini = S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0)
    assert rec.getExpectedValue(ini) == -17.800000000000008
    rows, _, _ = RO.reached_at(rec._m, [1], [[0.0] * 5])
    p2 = rows[rows[:, 0] == 2]
    for r in p2[np.linspace(0, len(p2) - 1, 40).astype(int)]:
        act = rec.getAction(S.CashStateMultiLead(2, *r[1:6]))
        assert (act.getFirstAction(), act.getSecondAction()) == (r[6], r[7])
    with pytest.raises(KeyError):
        rec.getAction(S.CashStateMultiLead(2, 1, 1, 1, 1, 0.123))
    n1 = sum(rec.n_states)
    late = S.CashStateMultiLead(2, 1, 1, 1, 1, 0.123)
    v = rec.getExpectedValue(late)
    want, vals, _ = RO.reached_at(rec._m, [1, 2], [[0.0] * 5, [1, 1, 1, 1, 0.123]])
    assert v == vals[1] and sum(rec.n_states) == len(want) == n1 + 1
    act = rec.getAction(late)
    row = want[(want[:, 0] == 2) & np.all(want[:, 1:6] == [1, 1, 1, 1, 0.123], axis=1)][0]
    assert (act.getFirstAction(), act.getSecondAction()) == (row[6], row[7])


@pytest.mark.gpu
def test_rounded_facade_opt_table_and_simulation(S):
    """CashConstraintTest.java:121-129 with the table and roll-out its CashRecursion gives: getOptTable() /
    getCacheActions() (CashRecursion.java:201-220) and CashSimulation(...).simulateSDPGivenSamplNum"""
    dists = [S.PoissonDist(m) for m in (6, 3, 2, 5)]
    rec, root = _rounded(S)
    ini = S.CashState(1, 0, 33.0)
    assert rec.getOptTable().shape == (0, 4)
    v = rec.getExpectedValue(ini)
    rows, vals, _ = RO.reached_at(rec._m, [1], [root])
    assert v == vals[0]
    tab = rec.getOptTable()
    assert np.array_equal(tab, rows[:, :4])
    acts = rec.getCacheActions()
    assert len(acts) == len(rows) and acts[S.CashState(1, 0, 33.0)] == rows[0][3]
    samples = S.generate_lh_samples(dists, 1000)
    sim = S.CashSimulation(dists, 1000, rec)
    got = sim.simulateSDPGivenSamplNum(ini, samples)
    want, memo, _ = RO.reached_simulate(rec._m, root, samples)
    assert got == float(want.sum() / len(want)) + 33.0
    assert np.array_equal(rec.getOptTable(), memo[:, :4])
    # a later-period state extends the handle
    late = S.CashState(3, 10.0, 12.34)
    lv = rec.getExpectedValue(late)
    st = [list(r[1:3]) for r in memo]
    pr = [int(r[0]) for r in memo]
    want, wv, _ = RO.reached_at(rec._m, pr + [3], st + [[10.0, 12.34]])
    assert lv == wv[-1] and np.array_equal(rec.getOptTable(), want[:, :4])
