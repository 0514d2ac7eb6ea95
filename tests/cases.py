"""Small instances of every model family: sizes the CPU oracle solves in about a second."""
from __future__ import annotations

import numpy as np

import sdpb200 as S
from sdpb200 import abi as A


def pmf(means, q=0.999):
    return S.poisson_pmf(means, q)


def two_point(T, lo, hi, p=0.5):
    """a pmf with non-consecutive demand values {lo, hi}"""
    return [np.array([[lo, p], [hi, 1 - p]], dtype=float) for _ in range(T)]


def case_A_small():
    return S.inventory_model(pmf([5, 8, 6]), fixed_cost=20, vari_cost=1, hold_cost=1, penalty_cost=5,
                             max_order=15, inv_min=-30, inv_max=30, name="A_small"), [[0.0]]


def case_A_max():
    # Recursion supports MAX (Recursion.java:44-47,152-157); same lambdas, maximised
    return S.inventory_model(pmf([3, 4]), fixed_cost=7, vari_cost=0.5, hold_cost=1.5, penalty_cost=4,
                             max_order=9, inv_min=-12, inv_max=14, direction=A.MAX, name="A_max"), [[2.0]]


def case_A_gy():
    return S.inventory_model(pmf([9, 23, 13], 0.9999), fixed_cost=500, vari_cost=0, hold_cost=2,
                             penalty_cost=10, max_order=30, inv_min=-80, inv_max=80, gy_mode=True,
                             name="A_gy"), [[1.0]]


def case_A_twopoint():
    # non-consecutive demand support and exact ties between actions
    return S.inventory_model(two_point(3, 4.0, 10.0), fixed_cost=0, vari_cost=0, hold_cost=1, penalty_cost=1,
                             max_order=12, inv_min=-20, inv_max=20, name="A_twopoint"), [[0.0]]


def case_A_halfstep():
    p = [np.array([[0.0, 0.25], [0.5, 0.25], [1.0, 0.25], [1.5, 0.25]]) for _ in range(3)]
    return S.inventory_model(p, fixed_cost=3, vari_cost=1, hold_cost=1, penalty_cost=9, max_order=4,
                             inv_min=-6, inv_max=6, step=0.5, name="A_halfstep"), [[0.0]]


def case_A_sparse_pmf():
    # generic DiscreteDistribution through GetPmf's cdf-difference branch (GetPmf.java:120-129): long
    # tables that are zero almost everywhere, as in fitss/LevelFitsS.java:66-71 (scaled down)
    values = [[3, 15, 28, 29], [1, 22, 23, 24], [1, 6, 12, 17]]
    probs = [[0.018, 0.888, 0.046, 0.048], [0.028, 0.271, 0.17, 0.531], [0.041, 0.027, 0.889, 0.043]]
    dists = [S.DiscreteDistribution(v, p) for v, p in zip(values, probs)]
    table = S.GetPmf(dists, 0.9999, 1).getpmf()
    return S.inventory_model(table, fixed_cost=50, vari_cost=0, hold_cost=1, penalty_cost=10, max_order=25,
                             inv_min=-60, inv_max=60, name="A_sparse_pmf"), [[0.0]]


def case_A_degenerate():
    # T = 1, a single action (order nothing), a single demand point
    return S.inventory_model([np.array([[2.0, 1.0]])], fixed_cost=5, vari_cost=1, hold_cost=1, penalty_cost=3,
                             max_order=0, inv_min=-3, inv_max=3, name="A_degenerate"), [[0.0]]


def case_A_one_state():
    # a grid of one inventory point: every successor clamps onto it
    return S.inventory_model(pmf([2, 3]), fixed_cost=1, vari_cost=1, hold_cost=1, penalty_cost=2, max_order=4,
                             inv_min=0, inv_max=0, name="A_one_state"), [[0.0]]


def case_B1_ref():
    # Leadtime.java:25-68 scaled down; unclamped, so the grid is the reachable hull
    T, mean, maxq = 3, 4, 12
    p = pmf([mean] * T)
    dmax = max(r[-1, 0] for r in p)
    return S.leadtime_model(p, fixed_cost=0, vari_cost=1, hold_cost=2, penalty_cost=10, max_order=maxq,
                            inv_min=-T * dmax, inv_max=T * maxq, lead_time=1, clamp=False,
                            name="B1_ref"), [[0.0, 0.0]]


def case_B1_fixed():
    return S.leadtime_model(pmf([4, 6, 5]), fixed_cost=15, vari_cost=1, hold_cost=2, penalty_cost=10,
                            max_order=10, inv_min=-25, inv_max=40, lead_time=1, clamp=True,
                            name="B1_fixed"), [[0.0, 0.0], [3.0, 2.0]]


def case_B2_small():
    return S.leadtime_model(pmf([3, 4, 3, 4]), fixed_cost=0, vari_cost=1, hold_cost=2, penalty_cost=10,
                            max_order=7, inv_min=-15, inv_max=15, lead_time=2, clamp=True,
                            name="B2_small"), [[0.0, 0.0, 0.0]]


def case_C_small():
    # CashConstraint.java:44-133 scaled down, 0.1 cash grid
    return S.cash_constraint_model(pmf([5, 5, 5]), price=10, vari_cost=1, salvage=0.5, max_order=12,
                                   inv_min=0, inv_max=25, cash_min=0, cash_max=120, name="C_small"), [[0.0, 10.0]]


def case_C_rich():
    # every optional term switched on: K, h, overhead, overhead rate, deposit rate, penalty, discount
    return S.cash_constraint_model(pmf([4, 6, 5]), price=6, vari_cost=2, fixed_cost=3, hold_cost=0.5,
                                   salvage=1.0, overhead=2, overhead_rate=0.125, deposit_rate=0.25,
                                   penalty_cost=0.5, max_order=9, inv_min=0, inv_max=20, cash_min=-20,
                                   cash_max=90, quantiser=A.Q_LONGDIV, q_mul=1.0, q_div=1.0, gamma=0.95,
                                   name="C_rich"), [[0.0, 20.0], [2.0, 5.0]]


def case_C_int():
    # CashConstraint.java:44-133 with the integer cash grid of CashConstraintTesting.java:146
    return S.cash_constraint_model(pmf([5, 6, 5, 4]), price=10, vari_cost=1, salvage=0.5, max_order=14,
                                   inv_min=0, inv_max=25, cash_min=0, cash_max=260, quantiser=A.Q_LONGDIV,
                                   q_mul=1.0, q_div=1.0, name="C_int"), [[0.0, 12.0]]


def case_C_int_tall():
    # 75 inventory rows, so that a shard of two or three spans several 8-row tiles of bi_cash_diag; not in ALL
    return S.cash_constraint_model(pmf([5, 6, 5]), price=10, vari_cost=1, salvage=0.5, max_order=14,
                                   inv_min=0, inv_max=74, cash_min=0, cash_max=120, quantiser=A.Q_LONGDIV,
                                   q_mul=1.0, q_div=1.0, name="C_int_tall"), [[0.0, 12.0]]


def case_C_int_K():
    # integer fixed cost / overhead / unit cost 2, negative cash allowed, discounting, inventory from 2
    return S.cash_constraint_model(pmf([4, 6, 5]), price=7, vari_cost=2, fixed_cost=3, salvage=1.0, overhead=2,
                                   max_order=11, inv_min=2, inv_max=19, cash_min=-15, cash_max=140,
                                   quantiser=A.Q_DIV, q_mul=1.0, q_div=1.0, gamma=0.9,
                                   name="C_int_K"), [[2.0, 20.0], [4.0, -3.0]]


def case_D_small():
    return S.cash_overdraft_model(pmf([6, 6, 6]), price=10, vari_cost=1, overhead_t=[20, 20, 20],
                                  od_limit=30, max_order=15, inv_min=0, inv_max=25, cash_min=-60,
                                  cash_max=150, name="D_small"), [[0.0, 0.0]]


def case_D_rich():
    return S.cash_overdraft_model(pmf([5, 7]), price=8, vari_cost=2, fixed_cost=4, salvage=1,
                                  overhead_t=[10, 15], r0=0.25, r2=0.125, r3=1.5, od_limit=20, interest_free=5,
                                  max_order=10, inv_min=0, inv_max=18, cash_min=-50, cash_max=100,
                                  quantiser=A.Q_DIV, q_mul=10.0, q_div=10.0, gamma=0.9,
                                  name="D_rich"), [[0.0, 10.0]]


def case_DL_small():
    # CashOverdraftLimit.java:30-99 scaled down; non-zero holding, deposit and salvage terms
    return S.cash_overdraft_limit_model(pmf([5, 6, 5]), price=8, vari_cost=2, fixed_cost=3, hold_cost=0.5,
                                        salvage=1, overhead_t=[6, 4, 5], interest_rate=0.125, deposit_rate=0.0625,
                                        max_order=9, inv_min=0, inv_max=18, cash_min=-40, cash_max=90,
                                        name="DL_small"), [[0.0, 5.0]]


def case_DT_small():
    # CashOverdraftTesting.java:30-120 scaled down
    return S.cash_overdraft_testing_model(pmf([4, 5, 4]), price=7, vari_cost=2, fixed_cost=2, hold_cost=0.5,
                                          interest_rate=0.2, min_cash_required=-10, max_order=8, inv_min=0,
                                          inv_max=16, cash_min=-30, cash_max=80, name="DT_small"), [[0.0, 6.0]]


def case_TP_small():
    # TestPaper.java:30-110 scaled down: uniform demand 0..6, rounding switched on from period 3
    table = S.GetPmf([S.UniformIntDist(0, 6)] * 4, 1, 1).getpmf()
    return S.cash_loan_model(table, price=10, vari_cost=2, hold_cost=1, deposit_rate=0.01, loan_rate=0.15,
                             salvage=5, min_cash_required=-20, max_order=10, inv_min=0, inv_max=30,
                             cash_min=-60, cash_max=120, round_from_period=3, q_mul=0.1, q_div=0.1,
                             name="TP_small"), [[0.0, 0.0]]


def case_E_small():
    # SingleProductLeadtime.java:28-119 scaled down; cash grid 0.5 instead of 0.01 to keep it small
    return S.cash_leadtime_model(pmf([4, 4, 4]), price=5, vari_cost=1, salvage=0.5, od_limit=40, max_order=8,
                                 inv_min=0, inv_max=16, cash_min=-40, cash_max=60, q_mul=2.0, q_div=2.0,
                                 name="E_small"), [[0.0, 0.0, 0.0]]


def case_F_small():
    # cashSurvival.java:51-147 scaled down
    T = 3
    return S.cash_survival_model(pmf([5, 7, 6], 0.99), price_t=[4, 5, 4], vari_cost_t=[1, 1, 2],
                                 overhead_t=[12, 10, 14], salvage=0.5, max_order=20, inv_min=0,
                                 inv_max=30, cash_min=-30, cash_max=120, name="F_small"), [[0.0, 15.0]]


def case_XR_small():
    # CashConstraintXR.java:34-110 scaled down (integer-valued Poisson table instead of Gamma)
    # (the order-up-to range is capped at 31 levels on purpose: the cap bites at visited states, which the model allows)
    spec = S.cash_xr_model(pmf([4, 4, 4], 0.99), price=4, vari_cost=2, salvage=1, max_order=30, inv_min=0,
                           inv_max=30, cash_min=-10, cash_max=90, name="XR_small")
    spec.allow = A.ALLOW_CAPPED_ACTIONS
    return spec, [[0.0, 30.0]]


def case_XR_uncapped():
    # the reference's own action set (CashConstraintXR.java:71-75 has no cap): max_order covers R_max / v
    return S.cash_xr_model(pmf([3, 3], 0.99), price=4, vari_cost=2, salvage=1, max_order=40, inv_min=0,
                           inv_max=20, cash_min=0, cash_max=40, name="XR_uncapped"), [[0.0, 20.0]]


def case_M2_small():
    # MultiItemCash.java:33-121 scaled down: two products, discrete demands (GetPmfMulti.java:158-171)
    d1 = S.DiscreteDistribution([1, 3, 4], [0.3, 0.5, 0.2])
    d2 = S.DiscreteDistribution([0, 2], [0.4, 0.6])
    table = S.GetPmfMulti([[d1] * 3, [d2] * 3], 0.999, 1).tables()
    return S.two_product_cash_model(table, price=(4, 9), vari_cost=(2, 4), salvage=(1, 1), q_bound=6, inv_max=9,
                                    cash_min=0, cash_max=70, name="M2_small"), [[0.0, 0.0, 12.0]]


def case_M2_poisson():
    # Poisson branch of GetPmfMulti, exact ties broken by the +0.1 tolerance, no tolerance variant below
    table = S.GetPmfMulti([[S.PoissonDist(1.5)] * 2, [S.PoissonDist(1.0)] * 2], 0.99, 1).tables()
    return S.two_product_cash_model(table, price=(5, 6), vari_cost=(2, 3), salvage=(1, 1.5), q_bound=5, inv_max=7,
                                    cash_min=0, cash_max=45, gamma=0.95, name="M2_poisson"), [[1.0, 0.0, 9.0]]


def case_W_small():
    # WorkforcePlanning.java:33-104 scaled down: binomial turnover depending on the hire-up-to level
    return S.workforce_model([0.5, 0.3, 0.4], fix_cost=30, unit_vari_cost=4, salary=6, unit_penalty=25,
                             min_staff=[8, 10, 6], max_hire=20, max_x=30, name="W_small"), [[0.0]]


# ---- terminal boundary function (FinalCash.BoundaryFuncton, CashRecursionV.java:125-128) ------------------
def case_A_terminal():
    # leftover stock is worth 0.75 per unit at the end of the horizon, backorders cost 2.5 per unit
    spec, init = case_A_small()
    spec.terminal_value = spec.tabulate(lambda x: -0.75 * np.maximum(x, 0) + 2.5 * np.maximum(-x, 0))
    spec.name = "A_terminal"
    return spec, init


def case_A_terminal_big():
    # enough states for the tiled kernels' multi-tile paths
    spec = S.inventory_model(pmf([7, 9, 8]), fixed_cost=12, vari_cost=1, hold_cost=1, penalty_cost=6, max_order=37,
                             inv_min=-1250, inv_max=1249, name="A_terminal_big")
    spec.terminal_value = spec.tabulate(lambda x: 0.125 * x * np.sin(x))
    return spec, [[0.0]]


def case_B2_terminal():
    spec, init = case_B2_small()
    spec.terminal_value = spec.tabulate(lambda x, q1, q2: -1.0 * np.maximum(x + q1 + q2, 0) + 3.0 * np.maximum(-x, 0))
    spec.name = "B2_terminal"
    return spec, init


def case_B1_terminal():
    spec, init = case_B1_fixed()
    spec.terminal_value = spec.tabulate(lambda x, q1: 0.5 * np.abs(x + q1))
    spec.name = "B1_terminal"
    return spec, init


def case_C_terminal():
    # MultiItemCashXW.java:118-121 form for one product: final cash plus the salvage value of the stock,
    # instead of the salvage term inside the immediate value
    spec = S.cash_constraint_model(pmf([5, 6, 5]), price=10, vari_cost=1, salvage=0.0, max_order=14, inv_min=0,
                                   inv_max=25, cash_min=0, cash_max=200, quantiser=A.Q_LONGDIV, q_mul=1.0, q_div=1.0,
                                   name="C_terminal")
    spec.terminal_value = spec.tabulate(lambda x, w: w + 0.5 * x)
    return spec, [[0.0, 12.0]]


def case_C_terminal_frac():
    spec, init = case_C_small()
    spec.terminal_value = spec.tabulate(lambda x, w: 0.25 * w + 0.5 * x)
    spec.name = "C_terminal_frac"
    return spec, init


def case_D_terminal():
    spec, init = case_D_small()
    spec.terminal_value = spec.tabulate(lambda x, w: np.minimum(w, 100.0) + 0.25 * x)
    spec.name = "D_terminal"
    return spec, init


def case_DL_terminal():
    spec, init = case_DL_small()
    spec.terminal_value = spec.tabulate(lambda x, w: w + 0.75 * x - 0.25 * np.maximum(-w, 0.0))
    spec.name = "DL_terminal"
    return spec, init


def case_DT_terminal():
    spec, init = case_DT_small()
    spec.terminal_value = spec.tabulate(lambda x, w: np.minimum(w, 60.0) + 0.5 * x)
    spec.name = "DT_terminal"
    return spec, init


def case_C_pen_div_terminal():
    # bankruptcy penalty and the round(w*10)/10 quantiser with long division (CashOverdraft.java:116's idiom) on the
    # cash-constraint lambdas
    spec = S.cash_constraint_model(pmf([4, 5, 4]), price=6, vari_cost=2, fixed_cost=2, hold_cost=0.5, salvage=0.0,
                                   overhead=1.5, penalty_cost=0.5, max_order=8, inv_min=0, inv_max=14, cash_min=-15,
                                   cash_max=60, quantiser=A.Q_LONGDIV, q_mul=10.0, q_div=10.0,
                                   name="C_pen_div_terminal")
    spec.terminal_value = spec.tabulate(lambda x, w: w + 0.5 * x)
    return spec, [[0.0, 10.0], [3.0, -4.0]]


def case_E_terminal():
    spec, init = case_E_small()
    spec.terminal_value = spec.tabulate(lambda x, w, q: w + 0.5 * (x + q))
    spec.name = "E_terminal"
    return spec, init


def case_M2_terminal():
    # MultiItemCashXW.java:118-121: boundFinalCash = cash + salPrice1 * x1 + salPrice2 * x2
    spec, init = case_M2_small()
    spec.salvage = 0.0
    spec.salvage2 = 0.0
    spec.terminal_value = spec.tabulate(lambda x1, x2, w: w + 1.0 * x1 + 2.0 * x2)
    spec.name = "M2_terminal"
    return spec, init


def case_W_terminal():
    spec, init = case_W_small()
    spec.terminal_value = spec.tabulate(lambda x: 3.0 * np.abs(x - 8.0))
    spec.name = "W_terminal"
    return spec, init


# ---- A(s) = {0} in the last period (SingleProductLeadtime.java:74-75) on the families with specialised kernels ----
def case_A_nolast():
    spec, init = case_A_small()
    spec.flags |= A.F_NO_ORDER_LAST
    spec.name = "A_nolast"
    return spec, init


def case_B2_nolast():
    spec, init = case_B2_small()
    spec.flags |= A.F_NO_ORDER_LAST
    spec.name = "B2_nolast"
    return spec, init


def case_C_int_nolast():
    spec, init = case_C_int()
    spec.flags |= A.F_NO_ORDER_LAST
    spec.name = "C_int_nolast"
    return spec, init


def case_CLSP_main():
    # src/capacitated/CLSP.java:196-272 scaled down: the inline pmf (no (int) cast, no LB = 0 override; the support
    # of Poisson(53) starts at 26), fixed cost, capacity; initial inventory 1
    table = S.clsp_inline_pmf([9, 23, 53, 29], 0.99999, 1)
    return S.inventory_model(table, fixed_cost=500, vari_cost=0, hold_cost=2, penalty_cost=10, max_order=60,
                             inv_min=-300, inv_max=300, name="CLSP_main"), [[1.0]]


NOLAST = [case_A_nolast, case_B2_nolast, case_C_int_nolast]

TERMINAL = [case_A_terminal, case_A_terminal_big, case_B1_terminal, case_B2_terminal, case_C_terminal,
            case_C_terminal_frac, case_D_terminal, case_DL_terminal, case_DT_terminal, case_C_pen_div_terminal,
            case_E_terminal, case_M2_terminal, case_W_terminal]

ALL = [case_A_small, case_A_max, case_A_gy, case_A_twopoint, case_A_halfstep, case_A_sparse_pmf,
       case_A_degenerate, case_A_one_state, case_B1_ref, case_B1_fixed,
       case_B2_small, case_C_small, case_C_rich, case_C_int, case_C_int_K, case_D_small, case_D_rich, case_DL_small,
       case_DT_small, case_TP_small, case_M2_small, case_M2_poisson, case_W_small, case_E_small, case_F_small,
       case_XR_small, case_XR_uncapped, case_CLSP_main] + TERMINAL + NOLAST


# ---- golden fixtures --------------------------------------------------------------------------
import os

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN = ["A_small", "A_gy", "A_twopoint", "B1_ref", "B2_small", "C_rich", "D_rich", "E_small", "F_small",
          "XR_small"]


def load_golden(name):
    """-> (spec with the pmf table stored in the fixture, init states, fixture dict)"""
    spec, init = globals()["case_" + name]()
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    lens = g["pmf_len"]
    off = np.concatenate([[0], np.cumsum(lens)])
    spec.pmf = [g["pmf"][off[i]:off[i + 1]] for i in range(len(lens))]
    return spec, init, g
