"""Host-side mirror of the reference's recursion engines, over libsdpb200.so.

Same class and member names as the Java classes (paths relative to /root/reference):

    State / Recursion                       src/sdp/inventory/State.java:12-71, Recursion.java:33-186
    LeadtimeState / LeadtimeRecursion       src/sdp/inventory/LeadtimeState.java:10-20, LeadtimeRecursion.java:20-102
    CashState / CashRecursion               src/sdp/cash/CashState.java:12-23, CashRecursion.java:24-220
    CashLeadtimeState / CashLeadtimeRecursion  src/sdp/cash/CashLeadtimeState.java:11-21, CashLeadtimeRecursion.java:20-105
    RiskState / RiskRecursion               src/sdp/cash/RiskState.java:12-26, RiskRecursion.java:24-135
    CashStateXR / CashRecursionXR           src/sdp/cash/CashStateXR.java:13-31, CashRecursionXR.java:24-150

The Java constructors take three lambdas (A, f, c).  A GPU cannot call them, so the constructors
here take a `ModelSpec` descriptor in their place (models.py lowers every in-scope reference driver
to one); the lambdas may still be passed as Python callables, in which case the descriptor is
spot-checked against them on random (state, action, demand) triples before anything is solved.

Behaviour kept from the reference: `getExpectedValue(state)` may be called for any state at any
time (the whole grid is solved on the first call — the GPU analogue of the lazy memoised solve);
`getAction(state)` on a state that was never solved raises (Java: NullPointerException from
unboxing, Recursion.java:165-167); `getOptTable()` returns only the states the top-down recursion
would have visited from the states queried so far, sorted by (period, state).
"""
from __future__ import annotations

import random
from enum import Enum

import ctypes as C

import numpy as np

from . import _abi as A
from .models import ModelSpec
from .solver import Reached, Solver, TopDown


class OptDirection(Enum):
    MIN = 0
    MAX = 1


# ---- states -------------------------------------------------------------------------------
class State:
    def __init__(self, period, iniInventory):
        self.period = int(period)
        self.initialInventory = float(iniInventory)

    def getPeriod(self):
        return self.period

    def getIniInventory(self):
        return self.initialInventory

    def _vec(self):
        return (self.initialInventory,)

    def _key(self):
        return (self.period,) + self._vec()

    def __eq__(self, o):
        return isinstance(o, State) and self._key() == o._key()

    def __hash__(self):
        return hash(self._key())

    def __repr__(self):
        return f"period = {self.period}, initialInventory = {self.initialInventory}"


class LeadtimeState(State):
    def __init__(self, period, iniInventory, preQ):
        super().__init__(period, iniInventory)
        self.preQ = float(preQ)

    def getPreQ(self):
        return self.preQ

    def _vec(self):
        return (self.initialInventory, self.preQ)


class CashState(State):
    def __init__(self, period, iniInventory, iniCash):
        super().__init__(period, iniInventory)
        self.iniCash = float(iniCash)

    def getIniCash(self):
        return self.iniCash

    def _vec(self):
        return (self.initialInventory, self.iniCash)


class CashLeadtimeState(CashState):
    def __init__(self, period, iniInventory, iniCash, preQ):
        super().__init__(period, iniInventory, iniCash)
        self.preQ = float(preQ)

    def getPreQ(self):
        return self.preQ

    def _vec(self):
        return (self.initialInventory, self.iniCash, self.preQ)


class RiskState(CashState):
    def __init__(self, period, iniInventory, iniCash, bankruptBefore=False):
        super().__init__(period, iniInventory, iniCash)
        self.bankruptBefore = False  # the reference constructor ignores its argument (RiskState.java:15-18)

    def getBankruptBefore(self):
        return self.bankruptBefore


class CashStateXR(State):
    def __init__(self, period, iniInventory, R, variCost):
        super().__init__(period, iniInventory)
        self.iniR = float(R)
        self.unitVariCost = float(variCost)

    def getIniR(self):
        return self.iniR

    def _vec(self):
        return (self.initialInventory, self.iniR)


# ---- engines ------------------------------------------------------------------------------
class _Engine:
    state_cls = State
    _kinds = (A.COST_BACKORDER,)
    _lead = 0

    def __init__(self, spec: ModelSpec, getFeasibleAction=None, stateTransition=None, immediateValue=None,
                 device: int = -1, kernel: int = A.KERNEL_AUTO, dedup: bool = False, spot_checks: int = 200,
                 boundFinalCash=None, allow: int = 0, devices=None, topdown: bool = False):
        """`boundFinalCash`: a FinalCash.BoundaryFuncton (src/sdp/inventory/FinalCash.java:16-18) -- a function of the
        state dimensions in API order, evaluated on numpy arrays over the whole grid (ModelSpec.tabulate) -- that
        values the states of period T+1 (CashRecursionV.java:125-128).  `allow`: sdpb_allow bits.  `devices`: a list
        of CUDA ordinals to partition the state grid over (sdpb_group_*); value queries work as usual, the visited-state
        tables (getOptTable) need a single-GPU engine.

        `topdown=True`: no grid.  The engine solves exactly the states the reference's recursion visits from the
        period-1 states asked for so far (sdpb_topdown_*), so states, steps and demands need not be multiples of a
        power of two and an unclamped model needs no hull; getExpectedValue on a new period-1 state solves only the
        states it reaches that no earlier call did (sdpb_topdown_extend), and a Simulation over this recursion adds
        the states its paths meet, as the reference's memo maps grow.  A later-period state that was not reached raises
        KeyError, as getAction on an unsolved state does.  The lambdas are kept but not spot-checked against the descriptor (that check evaluates them on
        the dense grid), and there is no boundary function (it is tabulated on the grid) and no multi-GPU split."""
        if spec.cost_kind not in self._kinds or spec.lead_time != self._lead:
            raise ValueError(f"{type(self).__name__} does not take this descriptor "
                             f"(cost_kind={spec.cost_kind}, lead_time={spec.lead_time})")
        self._topdown = topdown
        self._td = None
        if topdown:
            if boundFinalCash is not None or (devices is not None and len(devices) > 1):
                raise ValueError("topdown=True takes no boundFinalCash and runs on one GPU")
            self.spec, self.pmf = spec, spec.pmf
            self.getFeasibleActions, self.stateTransition, self.immediateValue = (getFeasibleAction, stateTransition,
                                                                                  immediateValue)
            self.boundFinalCash = None
            self._device, self._allow = device, allow
            self._queried = []
            self._tree_map = False
            return
        if boundFinalCash is not None:
            import copy
            spec = copy.copy(spec)
            spec.terminal_value = spec.tabulate(boundFinalCash)
        self.spec = spec
        self.pmf = spec.pmf
        self.getFeasibleActions = getFeasibleAction
        self.stateTransition = stateTransition
        self.immediateValue = immediateValue
        self.boundFinalCash = boundFinalCash
        self._group = None
        if devices is not None and len(devices) > 1:
            from .solver import Group
            self._group = Group(spec, list(devices), kernel=kernel, dedup=dedup, allow=allow)
            self._solver = self._group.shards[0]
        else:
            self._solver = Solver(spec, device=device if devices is None else devices[0], kernel=kernel, dedup=dedup,
                                  allow=allow)
        # dense-grid artefacts matter only at states the reference would visit (sdpb_allow): models that can have
        # them are checked from every queried period-1 state
        self._check_reach = (not (spec.flags & A.F_CLAMP_INV)) or spec.cost_kind == A.COST_CASH_XR
        self._solved = False
        self._queried = []  # period-1 states asked for so far: roots of the top-down visit set
        self._tree_map = False
        if immediateValue is not None or stateTransition is not None or getFeasibleAction is not None:
            self._spot_check(spot_checks)

    # -- the reference's accessors --
    def getStateTransitionFunction(self):
        return self.stateTransition

    def getImmediateValueFunction(self):
        return self.immediateValue

    def setTreeMapCacheAction(self):
        """Recursion.java:80-86: swaps the action map for a TreeMap with the same key order; a no-op
        here because tables are always produced in (period, state) order."""
        self._tree_map = True

    def _ensure_solved(self):
        if not self._solved:
            (self._group or self._solver).solve()
            self._solved = True

    def _value(self, state):
        if self._topdown:
            if self._td is None:
                raise KeyError(f"{state} was not reached: no period-1 state has been solved (Recursion.java:165-167)")
            try:
                v, q = self._td.value(state.getPeriod(), [state._vec()])
            except A.SdpbError as e:
                if e.code == A.SDPB_ERR_UNSOLVED:
                    raise KeyError(f"{state} was not reached from {self._queried} (Recursion.java:165-167)") from None
                raise
            return float(v[0]), float(q[0])
        self._ensure_solved()
        v, q = (self._group or self._solver).value(state.getPeriod(), [state._vec()])
        return float(v[0]), float(q[0])

    def getExpectedValue(self, state):
        if self._topdown:
            if state.getPeriod() == 1 and state._vec() not in self._queried:
                if self._td is None:
                    self._td = TopDown(self.spec, [state._vec()], device=self._device,
                                       allow=self._allow | self.spec.allow)
                else:
                    self._td.extend(1, [state._vec()])
                self._queried.append(state._vec())
            return self._value(state)[0]
        val, _ = self._value(state)
        if state.getPeriod() == 1 and state._vec() not in self._queried:
            self._queried.append(state._vec())
            if self._check_reach and self._group is None:
                # raises SDPB_ERR_OFFGRID if the dense grid clipped a successor (or capped the action set) of a state
                # the reference's recursion visits from here: the value would not be the reference's
                self._solver.reach(self._queried)
        return val

    def getAction(self, state):
        if self._topdown:
            return self._value(state)[1]
        if not self._solved:
            # Java: cacheActions.get(state) is null -> NullPointerException on unboxing
            raise KeyError("getAction on a state that was never solved (Recursion.java:165-167)")
        return self._value(state)[1]

    def getOptTable(self):
        """Rows [t, state dims..., Q*] for the visited states only (Recursion.java:177-186)."""
        if self._topdown:
            return self._td.opt_table() if self._td is not None else np.empty((0, self._ndim() + 2))
        if not self._queried:
            return np.empty((0, self._solver.ndim + 2))
        if self._group is not None:
            raise NotImplementedError("the visited-state table needs a single-GPU engine (sdpb_reach)")
        self._ensure_solved()
        self._solver.reach(self._queried)
        return self._solver.opt_table()

    def getCacheActions(self):
        """Map state -> optimal action over the visited states (Recursion.java:169-171)."""
        out = {}
        for row in self.getOptTable():
            out[self.state_cls(int(row[0]), *row[1:-1]) if self.state_cls is not CashStateXR
                else CashStateXR(int(row[0]), row[1], row[2], self.spec.vari_cost)] = float(row[-1])
        return out

    def stats(self):
        return self._td.stats() if self._topdown else self._solver.stats()

    def _ndim(self):
        return 1 + (self.spec.cost_kind != A.COST_BACKORDER) + self.spec.lead_time

    # -- descriptor <-> lambda validation --
    def _spot_check(self, n):
        """A descriptor/lambda mismatch would be silent, so compare them on random triples."""
        from . import _spot
        rng = random.Random(20261018)
        for _ in range(n):
            st, a, d = _spot.random_triple(self.spec, rng)
            state = self._make_state(st)
            c_desc, nxt_desc, nA = _spot.eval_descriptor(self.spec, st, a, d, solver=self._solver)
            if self.immediateValue is not None:
                c_user = float(self.immediateValue(state, a, d))
                if c_user != c_desc:
                    raise ValueError(f"descriptor and immediateValue lambda disagree at {state}, a={a}, d={d}: "
                                     f"{c_desc!r} vs {c_user!r}")
            if self.stateTransition is not None and st[0] < self.spec.T:
                nxt = self.stateTransition(state, a, d)
                if tuple(nxt._vec()) != tuple(nxt_desc):
                    raise ValueError(f"descriptor and stateTransition lambda disagree at {state}, a={a}, d={d}: "
                                     f"{nxt_desc} vs {nxt._vec()}")
            if self.getFeasibleActions is not None:
                if len(self.getFeasibleActions(state)) != nA:
                    raise ValueError(f"descriptor and getFeasibleAction lambda disagree at {state}")

    def _make_state(self, st):
        t, vec = st[0], st[1:]
        if self.state_cls is CashStateXR:
            return CashStateXR(t, vec[0], vec[1], self.spec.vari_cost)
        return self.state_cls(t, *vec)


class Recursion(_Engine):
    """new Recursion(OptDirection, pmf, A, f, c) -> Recursion(spec[, A, f, c]); Recursion.java:49-63."""
    OptDirection = OptDirection
    state_cls = State


class LeadtimeRecursion(_Engine):
    state_cls = LeadtimeState
    _lead = 1


class LeadtimeRecursion2(_Engine):
    """Lead time 2 (state (x, q1, q2)): the synthetic C4 extension; not a reference class."""
    _lead = 2

    class state_cls(State):  # noqa: N801
        def __init__(self, period, iniInventory, preQ, preQ2):
            super().__init__(period, iniInventory)
            self.preQ, self.preQ2 = float(preQ), float(preQ2)

        def _vec(self):
            return (self.initialInventory, self.preQ, self.preQ2)


class CashRecursion(_Engine):
    OptDirection = OptDirection
    state_cls = CashState
    _kinds = (A.COST_CASH_DEPOSIT, A.COST_CASH_OVERDRAFT, A.COST_CASH_OD_LIMIT, A.COST_CASH_OD_TESTING,
              A.COST_CASH_LOAN)

    def getSurvProb(self, state):
        """CashRecursion.java:143-194: needs a descriptor built with recursion=REC_SURVIVAL."""
        if self.spec.recursion != A.REC_SURVIVAL:
            raise ValueError("build the descriptor with recursion=REC_SURVIVAL to use getSurvProb")
        return self.getExpectedValue(state)


class RiskRecursion(CashRecursion):
    state_cls = RiskState

    def __init__(self, spec, *a, **k):
        if spec.recursion != A.REC_SURVIVAL:
            raise ValueError("RiskRecursion takes a REC_SURVIVAL descriptor (RiskRecursion.java:64-108)")
        super().__init__(spec, *a, **k)


class CashLeadtimeRecursion(_Engine):
    state_cls = CashLeadtimeState
    _kinds = (A.COST_CASH_DEPOSIT, A.COST_CASH_OVERDRAFT)
    _lead = 1


class CashRecursionXR(_Engine):
    OptDirection = OptDirection
    state_cls = CashStateXR
    _kinds = (A.COST_CASH_XR,)


# ---- two products ---------------------------------------------------------------------------
class CashStateMulti:
    """src/sdp/cash/multiItem/CashStateMulti.java:14-45."""

    def __init__(self, period, iniInventory1, iniInventory2, iniCash):
        self.period = int(period)
        self.iniInventory1, self.iniInventory2, self.iniCash = float(iniInventory1), float(iniInventory2), float(iniCash)

    def getPeriod(self):
        return self.period

    def getIniInventory1(self):
        return self.iniInventory1

    def getIniInventory2(self):
        return self.iniInventory2

    def getIniCash(self):
        return self.iniCash

    def _vec(self):
        return (self.iniInventory1, self.iniInventory2, self.iniCash)


class Actions:
    """src/sdp/cash/multiItem/Actions.java:17-33."""

    def __init__(self, action1, action2):
        self.firstAction, self.secondAction = int(action1), int(action2)

    def getFirstAction(self):
        return self.firstAction

    def getSecondAction(self):
        return self.secondAction

    def __eq__(self, o):
        return (self.firstAction, self.secondAction) == (o.firstAction, o.secondAction)

    def __repr__(self):
        return f"Actions({self.firstAction}, {self.secondAction})"


class CashRecursionMulti:
    """new CashRecursionMulti(discountFactor, pmf, buildActionList, f, c, T) ->
    CashRecursionMulti(spec); src/sdp/cash/multiItem/CashRecursionMulti.java:60-116."""

    def __init__(self, spec: ModelSpec, device: int = -1):
        if spec.cost_kind != A.COST_CASH_TWO_PRODUCT:
            raise ValueError("CashRecursionMulti takes a two-product descriptor")
        self.spec = spec
        self._solver = Solver(spec, device=device)
        self._solved = False

    def _value(self, state):
        if not self._solved:
            self._solver.solve()
            self._solved = True
        v, q = self._solver.value(state.getPeriod(), [state._vec()])
        n = self.spec.max_order_idx + 1
        return float(v[0]), Actions(int(q[0]) // n, int(q[0]) % n)

    def getExpectedValue(self, state):
        return self._value(state)[0]

    def getAction(self, state):
        if not self._solved:
            raise KeyError("getAction on a state that was never solved")
        return self._value(state)[1]

    def getOptTable(self, variCost, init_states):
        """CashRecursionMulti.getOptTable (CashRecursionMulti.java:187-209): rows
        [period, x1, x2, w, R, boolAlpha, alpha, Q1, Q2, c1, c2] over the states the recursion visits
        from `init_states` (period-1 states (x1, x2, w))."""
        if not self._solved:
            self._solver.solve()
            self._solved = True
        self._solver.reach(init_states)
        n = self.spec.max_order_idx + 1
        out = []
        for t, x1, x2, w, q in self._solver.opt_table():
            Q1, Q2 = float(int(q) // n), float(int(q) % n)
            R = w + x1 * variCost[0] + x2 * variCost[1]
            boolAlpha, alpha = 0.0, 10000.0
            if w <= variCost[0] * Q1 + variCost[1] * Q2 and Q1 > 0 and Q2 > 0:
                boolAlpha, alpha = 1.0, variCost[0] * Q1 / w
            out.append([t, x1, x2, w, R, boolAlpha, alpha, Q1, Q2, variCost[0], variCost[1]])
        return np.asarray(out)


class CashStateMultiLead:
    """src/sdp/cash/multiItem/CashStateMultiLead.java: (period, iniInventory1, iniInventory2, preQ1, preQ2, iniCash)."""

    def __init__(self, period, iniInventory1, iniInventory2, preQ1, preQ2, iniCash):
        self.period = int(period)
        self.iniInventory1, self.iniInventory2 = float(iniInventory1), float(iniInventory2)
        self.preQ1, self.preQ2, self.iniCash = float(preQ1), float(preQ2), float(iniCash)

    def getPeriod(self):
        return self.period

    def _vec(self):
        return (self.iniInventory1, self.iniInventory2, self.preQ1, self.preQ2, self.iniCash)


class _ReachedEngine:
    """The two-product engines whose states do not live on a grid: solved over the states the reference's recursion
    reaches from the states queried so far, kept in one handle (sdpb_reached_*): getAction answers every reached state,
    and a Simulation / CashSimulation over the engine rolls its policy out.  `pmf`: per period an array [D, 3] of
    (demand1, demand2, prob) as GetPmfMulti.getPmf returns."""
    kind = A.REACHED_MULTILEAD

    def _setup(self, pmf, price, variCost, salvage, overheadCost, Qbound, minInventoryState, maxInventoryState,
               minCashState, maxCashState, discountFactor, tieTolerance, device, depositeRate=0.0, r0=0.0, r1=0.0, r2=0.0,
               limit=0.0, interestFreeAmount=0.0, fixedCost=0.0, holdingCost=0.0, minCashRequired=0.0, stateQ=0.0):
        self.lib = A.load()
        T = len(pmf)
        lens = [len(r) for r in pmf]
        nD = max(lens)
        tab = np.zeros((T, nD, 3))                                                # [T, D, 3], shorter periods padded
        for t, r in enumerate(pmf):
            r = np.asarray(r, dtype=np.float64)
            if r.shape[1] == 2:                                                   # one product: (demand, prob)
                r = np.column_stack([r[:, 0], np.zeros(len(r)), r[:, 1]])
            tab[t, :len(r)] = r
        self._lens = np.ascontiguousarray(lens, dtype=np.int32)
        self._d1 = np.ascontiguousarray(tab[:, :, 0]).ravel()
        self._d2 = np.ascontiguousarray(tab[:, :, 1]).ravel()
        self._p = np.ascontiguousarray(tab[:, :, 2]).ravel()
        self._ovh = np.ascontiguousarray(overheadCost if overheadCost is not None else [0.0] * T, dtype=np.float64)
        m = A.SdpbReachedModel()
        m.struct_size = C.sizeof(A.SdpbReachedModel)
        m.kind, m.T, m.q_bound, m.n_demands = self.kind, T, int(Qbound), nD
        dp = C.POINTER(C.c_double)
        m.d1, m.d2, m.p = self._d1.ctypes.data_as(dp), self._d2.ctypes.data_as(dp), self._p.ctypes.data_as(dp)
        m.overhead_t = self._ovh.ctypes.data_as(dp)
        m.price[0], m.price[1] = price
        m.vari_cost[0], m.vari_cost[1] = variCost
        m.salvage[0], m.salvage[1] = salvage
        m.r0, m.r1, m.r2, m.limit, m.interest_free = r0, r1, r2, limit, interestFreeAmount
        m.deposit_rate = depositeRate
        m.min_inv, m.max_inv, m.min_cash, m.max_cash = minInventoryState, maxInventoryState, minCashState, maxCashState
        m.gamma, m.tie_tolerance = discountFactor, tieTolerance
        m.fixed_cost, m.hold_cost, m.min_cash_required, m.state_q = fixedCost, holdingCost, minCashRequired, stateQ
        m.n_demands_t = self._lens.ctypes.data_as(C.POINTER(C.c_int32))
        self._m, self.T, self.device = m, T, device
        self._rh = None      # the Reached handle: one memo for every getExpectedValue call
        self._asked = set()  # (period, state) pairs getExpectedValue has been called on
        self.n_states = None
        self.solve_ms = None

    def _value(self, state):
        if self._rh is None:
            raise KeyError(f"{state._vec()} was not reached: getExpectedValue has not been called")
        try:
            v, a1, a2 = self._rh.value(state.getPeriod(), [state._vec()])
        except A.SdpbError as e:
            if e.code == A.SDPB_ERR_UNSOLVED:
                raise KeyError(f"getAction on a state that was never reached: period {state.getPeriod()}, "
                               f"{state._vec()}") from None
            raise
        return float(v[0]), (float(a1[0]), float(a2[0]))

    def getExpectedValue(self, state):
        """A state of any period: the first call on it extends the one memo with the states it reaches (only those no
        earlier call reached are solved); n_states / solve_ms then describe the memo and that call."""
        key = (state.getPeriod(), state._vec())
        if key not in self._asked:
            if self._rh is None:
                self._rh = Reached(self._m, [], device=self.device)
            self._rh.extend(*key)
            self._asked.add(key)
            self.n_states, self.solve_ms = self._rh.n_states(), self._rh.stats()["solve_ms"]
        return self._value(state)[0]

    def _action(self, state):
        return self._value(state)[1]


class CashRecursionMultiLead(_ReachedEngine):
    """new CashRecursionMultiLead(discountFactor, PmfMulti, buildActionList, stateTransition, immediateValue, T)
    (src/sdp/cash/multiItem/CashRecursionMultiLead.java:28-95) for the lambdas of
    src/cash/overdraft/MultiProductLeadtime.java:150-224: two products, lead time 1, overdraft interest, a cash balance
    that is NOT quantised."""
    kind = A.REACHED_MULTILEAD

    def __init__(self, pmf, price=(5.0, 10.0), variCost=(1.0, 2.0), salValueUnit=None, overheadCost=None, r0=0.0, r1=0.1,
                 r2=2.0, limit=500.0, interestFreeAmount=0.0, Qbound=50, minInventoryState=0.0, maxInventoryState=200.0,
                 minCashState=-500.0, maxCashState=5000.0, discountFactor=1.0, tieTolerance=0.1, device: int = -1):
        sal = salValueUnit if salValueUnit is not None else (variCost[0] * 0.5, variCost[1] * 0.5)
        self._setup(pmf, price, variCost, sal, overheadCost if overheadCost is not None else [100.0] * len(pmf), Qbound,
                    minInventoryState, maxInventoryState, minCashState, maxCashState, discountFactor, tieTolerance, device,
                    r0=r0, r1=r1, r2=r2, limit=limit, interestFreeAmount=interestFreeAmount)

    def getAction(self, state):
        a = self._action(state)
        return Actions(int(a[0]), int(a[1]))


class CashStateMultiXR:
    """src/sdp/cash/multiItem/CashStateMultiXR.java: (period, iniInventory1, iniInventory2, iniR)."""

    def __init__(self, period, iniInventory1, iniInventory2, iniR):
        self.period = int(period)
        self.iniInventory1, self.iniInventory2, self.iniR = float(iniInventory1), float(iniInventory2), float(iniR)

    def getPeriod(self):
        return self.period

    def _vec(self):
        return (self.iniInventory1, self.iniInventory2, self.iniR)


class CashRecursionMultiXR(_ReachedEngine):
    """new CashRecursionMultiXR(discountFactor, PmfMulti, buildActionList, stateTransition, immediateValue, T)
    (src/sdp/cash/multiItem/CashRecursionMultiXR.java:39-95) for the lambdas of
    src/cash/multiItem/MultiItemCashXR.java:73-126: state (x1, x2, R = w + v.x), actions = order-up-to pairs;
    getAction returns the pair of order-up-to levels (double[] in the reference)."""
    kind = A.REACHED_MULTI_XR

    def __init__(self, pmf, price=(5.0, 10.0), variCost=(1.0, 2.0), salPrice=None, depositeRate=0.0, Qbound=50,
                 minInventoryState=0.0, maxInventoryState=200.0, minCashState=0.0, maxCashState=10000.0, discountFactor=1.0,
                 tieTolerance=0.1, device: int = -1):
        sal = salPrice if salPrice is not None else (variCost[0] * 0.5, variCost[1] * 0.5)
        self._setup(pmf, price, variCost, sal, None, Qbound, minInventoryState, maxInventoryState, minCashState,
                    maxCashState, discountFactor, tieTolerance, device, depositeRate=depositeRate)

    def getAction(self, state):
        return list(self._action(state))


class CashRecursionRounded(_ReachedEngine):
    """new CashRecursion(OptDirection.MAX, pmf, getFeasibleAction, stateTransition, immediateValue, discountFactor)
    (src/sdp/cash/CashRecursion.java:39-140) for the lambdas of src/cash/singleItem/CashConstraintTest.java:76-116:
    one product, both state components rounded as Math.round(v * 0.1) / 0.1 after every transition (inventory
    levels such as 30.000000000000004: no axis with an exact step), an initial cash that need not be rounded
    (iniCash = 33).  Solved over the reached states.  State: CashState; getAction returns the order quantity."""
    kind = A.REACHED_CASH_ROUNDED

    def __init__(self, pmf, price=4.0, variCost=1.0, fixOrderCost=24.0, holdingCost=0.0, salvageValue=0.0,
                 interestRate=0.0, minCashRequired=0.0, maxOrderQuantity=200, minInventoryState=0.0,
                 maxInventoryState=500.0, minCashState=-100.0, maxCashState=2000.0, discountFactor=1.0, stateQ=0.1,
                 device: int = -1):
        self._setup(pmf, (price, 0.0), (variCost, 0.0), (salvageValue, 0.0), None, int(maxOrderQuantity) + 1,
                    minInventoryState, maxInventoryState, minCashState, maxCashState, discountFactor, 0.0, device,
                    depositeRate=interestRate, fixedCost=fixOrderCost, holdingCost=holdingCost,
                    minCashRequired=minCashRequired, stateQ=stateQ)

    def getAction(self, state):
        return self._action(state)[0]

    def getOptTable(self):
        """CashRecursion.java:201-220: rows [t, x, w, Q] of every reached state in memo-map order."""
        if self._rh is None:
            return np.empty((0, 4))
        return self._rh.opt_table()[:, :4]

    def getCacheActions(self):
        """Map CashState -> order quantity over the reached states."""
        return {CashState(int(t), x, w): float(q) for t, x, w, q in self.getOptTable()}


class CashRecursionV(_ReachedEngine):
    """new CashRecursionV(discountFactor, PmfMulti, buildActionListV, buildActionListPai, stateTransition,
    boundFinalCash, T, variCost) (src/sdp/cash/multiItem/CashRecursionV.java:47-131) for the lambdas of
    src/cash/multiItem/MultiItemYR.java:89-146: V(x1, x2, w) = max over affordable order-up-to pairs of
    Pi(y1, y2, R) = E V_{t+1}; the states of period T+1 are valued by the boundary function
    boundFinalCash(s) = w + salPrice . x (FinalCash.BoundaryFuncton).  State: CashStateMulti."""
    kind = A.REACHED_MULTI_YR

    def __init__(self, pmf, price=(5.0, 10.0), variCost=(1.0, 2.0), salPrice=None, depositeRate=0.0, Qbound=50,
                 minInventoryState=0.0, maxInventoryState=200.0, minCashState=0.0, maxCashState=10000.0, discountFactor=1.0,
                 tieTolerance=0.01, device: int = -1):
        sal = salPrice if salPrice is not None else (variCost[0] * 0.5, variCost[1] * 0.5)
        self._setup(pmf, price, variCost, sal, None, Qbound, minInventoryState, maxInventoryState, minCashState,
                    maxCashState, discountFactor, tieTolerance, device, depositeRate=depositeRate)

    def getExpectedValueV(self, state):
        return self.getExpectedValue(state)

    def getAction(self, state):
        return list(self._action(state))


# ---- workforce ------------------------------------------------------------------------------
class StaffState(State):
    """src/workforce/StaffState.java:4-14."""

    def __init__(self, period, iniStaffNum):
        super().__init__(period, iniStaffNum)
        self.iniStaffNum = int(iniStaffNum)


class StaffRecursion(_Engine):
    """new StaffRecursion(A, f, c, pmf, T) -> StaffRecursion(spec); src/workforce/StaffRecursion.java:39-121.
    getOptTable() rows are [t, staff, hires] (StaffRecursion.java:274-283); lambda spot checks are not wired
    for this kind."""
    state_cls = StaffState
    _kinds = (A.COST_STAFF,)

    def getAction(self, state):
        return int(super().getAction(state))
