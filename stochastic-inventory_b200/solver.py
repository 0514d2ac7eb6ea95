"""`Solver`: one sdpb_handle.  Thin, typed access to the C-ABI; all compute happens in
libsdpb200.so on the GPU.  Nothing here can solve anything on the CPU."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi as A
from .models import ModelSpec


def make_options(device=-1, shard_rank=0, shard_count=1, kernel=A.KERNEL_AUTO, dedup=False, stream=None, allow=0,
                 strict_cash_bounds=False, profile=False):
    opt = A.SdpbOptions()
    opt.struct_size = C.sizeof(A.SdpbOptions)
    opt.device, opt.shard_rank, opt.shard_count = device, shard_rank, shard_count
    opt.kernel, opt.dedup = kernel, 1 if dedup else 0
    opt.stream = stream
    opt.allow, opt.strict_cash_bounds, opt.profile = allow, 1 if strict_cash_bounds else 0, 1 if profile else 0
    return opt


def reachable_hull(spec: ModelSpec, init_states):
    """(inv_lo, inv_hi): inventory interval containing every state the reference's top-down recursion can visit
    from `init_states` (sdpb_reachable_hull; host arithmetic, needs no GPU) -- the grid an unclamped model needs."""
    lib = A.load()
    st = np.ascontiguousarray(np.atleast_2d(np.asarray(init_states, dtype=np.float64)))
    lo, hi = C.c_double(), C.c_double()
    m = spec.to_struct()
    rc = lib.sdpb_reachable_hull(C.byref(m), st.ctypes.data_as(C.POINTER(C.c_double)), st.shape[0],
                                 C.byref(lo), C.byref(hi))
    if rc != A.SDPB_OK:
        raise A.SdpbError(rc, "sdpb_reachable_hull")
    return lo.value, hi.value


def solve_batch(solvers):
    """Solve many independent small instances together (sdpb_solve_batch: one CUDA graph from the second call on)."""
    lib = A.load()
    arr = (C.c_void_p * len(solvers))(*[s.h for s in solvers])
    rc = lib.sdpb_solve_batch(arr, len(solvers))
    if rc != A.SDPB_OK:
        raise A.SdpbError(rc, lib.sdpb_last_error(solvers[0].h).decode())


class Solver:
    def __init__(self, spec: ModelSpec, device: int = -1, shard_rank: int = 0, shard_count: int = 1,
                 kernel: int = A.KERNEL_AUTO, dedup: bool = False, stream: int | None = None, allow: int = 0,
                 strict_cash_bounds: bool = False, profile: bool = False):
        self.lib = A.load()
        self.spec = spec
        self._model = spec.to_struct()
        opt = make_options(device, shard_rank, shard_count, kernel, dedup, stream, allow | spec.allow,
                           strict_cash_bounds, profile)
        h = C.c_void_p()
        rc = self.lib.sdpb_create(C.byref(self._model), C.byref(opt), C.byref(h))
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_last_error(None).decode())
        self.h = h
        g = A.SdpbGrid()
        self._check(self.lib.sdpb_grid_info(self.h, C.byref(g)))
        self.grid = g
        self.ndim = g.ndim
        self.n_states = g.n_states
        self.T = g.T

    def _check(self, rc):
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.sdpb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- solve ----
    def solve(self):
        self._check(self.lib.sdpb_solve(self.h))
        return self

    def solve_async(self):
        """Enqueue the whole solve on the handle's stream (CUDA-graph replay from the second call)."""
        self._check(self.lib.sdpb_solve_async(self.h))

    def solve_period_async(self, period: int):
        self._check(self.lib.sdpb_solve_period_async(self.h, period))

    def sync(self):
        self._check(self.lib.sdpb_sync(self.h))

    # ---- results ----
    def value(self, period: int, states):
        """(V, Q) for an array of API-order states [n, ndim]."""
        st = np.ascontiguousarray(np.atleast_2d(np.asarray(states, dtype=np.float64)))
        if st.shape[1] != self.ndim:
            raise ValueError(f"states must have {self.ndim} columns")
        n = st.shape[0]
        v = np.empty(n)
        q = np.empty(n)
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_value(self.h, period, st.ctypes.data_as(dp), n,
                                        v.ctypes.data_as(dp), q.ctypes.data_as(dp)))
        return v, q

    def period_tables(self, period: int, want_q: bool = True, out_v=None, out_q=None):
        """Whole-grid V_t and order quantities.  `out_v` / `out_q`: caller-owned float64 arrays of n_states
        (e.g. views of page-locked memory, which the device copies into at PCIe speed)."""
        dp = C.POINTER(C.c_double)
        for o in (out_v, out_q):
            if o is not None and (o.dtype != np.float64 or o.size != self.n_states or not o.flags.c_contiguous):
                raise ValueError("output buffers must be contiguous float64 arrays of n_states")
        V = out_v if out_v is not None else np.empty(self.n_states)
        Q = (out_q if out_q is not None else np.empty(self.n_states)) if want_q else None
        self._check(self.lib.sdpb_period_tables(self.h, period, V.ctypes.data_as(dp),
                                                Q.ctypes.data_as(dp) if want_q else None))
        return V, Q

    def shard_tables(self, period: int, want_q: bool = True):
        """This shard's block [shard_lo, shard_hi) of V_t and the order quantities."""
        n = self.grid.shard_hi - self.grid.shard_lo
        dp = C.POINTER(C.c_double)
        V = np.empty(n)
        Q = np.empty(n) if want_q else None
        self._check(self.lib.sdpb_shard_tables(self.h, period, V.ctypes.data_as(dp),
                                               Q.ctypes.data_as(dp) if want_q else None))
        return V, Q

    # ---- multi-GPU: shards of one model, connected through peer-mapped memory ----
    def peer_export(self) -> bytes:
        buf = C.create_string_buffer(A.PEER_BLOB_BYTES)
        self._check(self.lib.sdpb_peer_export(self.h, buf))
        return buf.raw

    def peer_attach(self, blobs):
        """`blobs`: every shard's peer_export(), in rank order."""
        raw = b"".join(blobs)
        self._check(self.lib.sdpb_peer_attach(self.h, C.c_char_p(raw), len(blobs)))

    def peer_traffic(self):
        a, b = C.c_int64(), C.c_int64()
        self._check(self.lib.sdpb_peer_traffic(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def period_profile(self):
        """[T, 3] device ms of the last sharded solve: kernels, pushes + flag, wait for the peers (profile=True)."""
        out = np.empty((self.T, 3))
        self._check(self.lib.sdpb_period_profile(self.h, out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def device_tables(self, period: int):
        dv, dq = C.c_void_p(), C.c_void_p()
        self._check(self.lib.sdpb_device_tables(self.h, period, C.byref(dv), C.byref(dq)))
        return dv.value, dq.value

    def shard_reads(self):
        """[lo, hi) of the flattened V_{t+1} this shard's kernels may read (multi-GPU halo exchange)."""
        lo, hi = C.c_int64(), C.c_int64()
        self._check(self.lib.sdpb_shard_reads(self.h, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def state_of_index(self, idx: int):
        st = np.empty(self.ndim)
        self._check(self.lib.sdpb_state_of_index(self.h, idx, st.ctypes.data_as(C.POINTER(C.c_double))))
        return st

    def reach(self, init_states):
        st = np.ascontiguousarray(np.atleast_2d(np.asarray(init_states, dtype=np.float64)))
        self._check(self.lib.sdpb_reach(self.h, st.ctypes.data_as(C.POINTER(C.c_double)), st.shape[0]))

    def opt_table(self):
        n = C.c_size_t(0)
        self._check(self.lib.sdpb_opt_table(self.h, None, C.byref(n)))
        rows = np.empty((n.value, self.ndim + 2))
        self._check(self.lib.sdpb_opt_table(self.h, rows.ctypes.data_as(C.POINTER(C.c_double)), C.byref(n)))
        return rows

    def simulate(self, init_state, samples, discount: float = 1.0):
        """Roll the solved policy over demand sample paths [n, T] -> per-path sums (Simulation.java:59-70)."""
        st = np.ascontiguousarray(init_state, dtype=np.float64)
        sm = np.ascontiguousarray(samples, dtype=np.float64)
        if sm.ndim != 2 or sm.shape[1] != self.T:
            raise ValueError(f"samples must be [n, {self.T}]")
        vals = np.empty(sm.shape[0])
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_simulate(self.h, st.ctypes.data_as(dp), sm.ctypes.data_as(dp), sm.shape[0],
                                           float(discount), vals.ctypes.data_as(dp)))
        return vals

    def stats(self):
        s = A.SdpbStats()
        self._check(self.lib.sdpb_stats_get(self.h, C.byref(s)))
        return {"evals": s.evals, "solve_ms": s.solve_ms, "kernel_ms": s.kernel_ms,
                "launches": s.launches, "kernel_used": s.kernel_used, "fp64_ops": s.fp64_ops,
                "evals_executed": s.evals_executed, "clipped_successors": s.clipped_successors,
                "capped_action_sets": s.capped_action_sets, "cash_bound_hits": s.cash_bound_hits,
                "exchange_ms": s.exchange_ms}


class TopDown:
    """One sdpb_topdown handle: `spec` solved over the states its top-down recursion reaches from the period-1 states
    `init_states` ([n, ndim], API order).  Needs no grid: states, steps and demands need not be multiples of a power of
    two, and an unclamped model needs no hull.  `scratch_bytes` bounds the forward expansion (0 = a fraction of free
    device memory).  Release the device memory with close() (or use it as a context manager)."""

    def __init__(self, spec: ModelSpec, init_states, device=None, allow=None, scratch_bytes: int = 0):
        self.lib = A.load()
        self.spec = spec
        self._model = spec.to_struct()
        self.ndim = 1 + (spec.cost_kind != A.COST_BACKORDER) + spec.lead_time
        self.T = spec.T
        st = np.ascontiguousarray(np.atleast_2d(np.asarray(init_states, dtype=np.float64)))
        if st.shape[1] != self.ndim:
            raise ValueError(f"initial states must have {self.ndim} columns")
        opt = A.SdpbTopdownOptions()
        opt.struct_size = C.sizeof(A.SdpbTopdownOptions)
        opt.device = -1 if device is None else device
        opt.allow = spec.allow if allow is None else allow
        opt.scratch_bytes = scratch_bytes
        h = C.c_void_p()
        rc = self.lib.sdpb_topdown_solve(C.byref(self._model), C.byref(opt), st.ctypes.data_as(C.POINTER(C.c_double)),
                                         st.shape[0], C.byref(h))
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_topdown_last_error(None).decode())
        self.h = h

    def _check(self, rc):
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_topdown_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.sdpb_topdown_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def value(self, period: int, states):
        """(V, Q) of reached API-order states [n, ndim] of one period; SDPB_ERR_UNSOLVED for a state not reached."""
        st = np.ascontiguousarray(np.atleast_2d(np.asarray(states, dtype=np.float64)))
        if st.shape[1] != self.ndim:
            raise ValueError(f"states must have {self.ndim} columns")
        n = st.shape[0]
        v, q = np.empty(n), np.empty(n)
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_topdown_value(self.h, period, st.ctypes.data_as(dp), n, v.ctypes.data_as(dp),
                                                q.ctypes.data_as(dp)))
        return v, q

    def extend(self, period: int, states):
        """getExpectedValue on API-order states [n, ndim] of one period: solves only the states no earlier call reached
        (sdpb_topdown_extend).  A failure leaves the handle as it was."""
        st = np.ascontiguousarray(np.atleast_2d(np.asarray(states, dtype=np.float64)))
        if st.shape[1] != self.ndim:
            raise ValueError(f"states must have {self.ndim} columns")
        self._check(self.lib.sdpb_topdown_extend(self.h, period, st.ctypes.data_as(C.POINTER(C.c_double)), st.shape[0]))
        return self

    def simulate(self, init_state, samples, discount: float = 1.0):
        """Roll the policy over demand sample paths [n, T] -> per-path sums (Simulation.java:59-70), solving every state
        a path meets that was not reached yet, as the reference's getExpectedValue at each step does
        (sdpb_topdown_simulate).  The states it adds stay in the handle."""
        st = np.ascontiguousarray(init_state, dtype=np.float64)
        sm = np.ascontiguousarray(samples, dtype=np.float64)
        if st.shape != (self.ndim,):
            raise ValueError(f"init_state must have {self.ndim} components")
        if sm.ndim != 2 or sm.shape[1] != self.T:
            raise ValueError(f"samples must be [n, {self.T}]")
        vals = np.empty(sm.shape[0])
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_topdown_simulate(self.h, st.ctypes.data_as(dp), sm.ctypes.data_as(dp), sm.shape[0],
                                                   float(discount), vals.ctypes.data_as(dp)))
        return vals

    def opt_table(self):
        """[rows, ndim + 2]: (t, state..., Q*) of every reached state in memo-map order."""
        n = C.c_size_t(0)
        self._check(self.lib.sdpb_topdown_opt_table(self.h, None, C.byref(n)))
        rows = np.empty((n.value, self.ndim + 2))
        self._check(self.lib.sdpb_topdown_opt_table(self.h, rows.ctypes.data_as(C.POINTER(C.c_double)), C.byref(n)))
        return rows

    def n_states(self):
        """Reached states of each period (T entries)."""
        out = (C.c_int64 * self.T)()
        self._check(self.lib.sdpb_topdown_states(self.h, out))
        return list(out)

    def stats(self):
        s = A.SdpbStats()
        self._check(self.lib.sdpb_topdown_stats(self.h, C.byref(s)))
        return {"evals": s.evals, "solve_ms": s.solve_ms, "kernel_ms": s.kernel_ms, "launches": s.launches,
                "capped_action_sets": s.capped_action_sets}


class Reached:
    """One sdpb_reached handle: a two-product (or CashConstraintTest) model, an `SdpbReachedModel`, solved over the
    states its recursion reaches from the period-1 states `init_states` ([n, ndim], API order; none gives an empty
    handle).  Every reached state can be queried, the handle extended with states of any period, and the policy rolled
    out over sample paths.  `scratch_bytes` > 0 replaces the free device memory as the expansion budget.  The model's
    tables are copied at construction.  Release the device memory with close() (or use it as a context manager)."""
    _NDIM = {A.REACHED_MULTILEAD: 5, A.REACHED_MULTI_XR: 3, A.REACHED_MULTI_YR: 3, A.REACHED_CASH_ROUNDED: 2}

    def __init__(self, model, init_states=(), device: int = -1, scratch_bytes: int = 0):
        self.lib = A.load()
        self.ndim = self._NDIM[model.kind]
        self.nd = 1 if model.kind == A.REACHED_CASH_ROUNDED else 2  # demands per period of a sample path
        self.T = model.T
        st = self._states(init_states)
        h = C.c_void_p()
        rc = self.lib.sdpb_reached_open(C.byref(model), device, scratch_bytes, st.ctypes.data_as(C.POINTER(C.c_double)),
                                        st.shape[0], C.byref(h))
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_reached_last_error().decode())
        self.h = h

    def _states(self, states):
        return np.ascontiguousarray(np.asarray(states, dtype=np.float64).reshape(-1, self.ndim))

    def _check(self, rc):
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_reached_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.sdpb_reached_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def value(self, period: int, states):
        """(V, a1, a2) of reached API-order states [n, ndim] of one period; SDPB_ERR_UNSOLVED for a state not reached."""
        st = self._states(states)
        n = st.shape[0]
        v, a1, a2 = np.empty(n), np.empty(n), np.empty(n)
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_reached_value(self.h, period, st.ctypes.data_as(dp), n, v.ctypes.data_as(dp),
                                                a1.ctypes.data_as(dp), a2.ctypes.data_as(dp)))
        return v, a1, a2

    def extend(self, period: int, states):
        """getExpectedValue on API-order states [n, ndim] of one period: solves only the states no earlier call reached.
        A failure leaves the handle as it was."""
        st = self._states(states)
        self._check(self.lib.sdpb_reached_extend(self.h, period, st.ctypes.data_as(C.POINTER(C.c_double)), st.shape[0]))
        return self

    def simulate(self, init_state, samples, discount: float = 1.0):
        """Roll the policy over demand sample paths [n, T, nd] (nd = 2 for two products; [n, T] for one) -> per-path
        sums, solving every state a path meets that was not reached yet.  The states it adds stay in the handle."""
        st = np.ascontiguousarray(init_state, dtype=np.float64)
        sm = np.ascontiguousarray(samples, dtype=np.float64)
        if st.shape != (self.ndim,):
            raise ValueError(f"init_state must have {self.ndim} components")
        if self.nd == 1 and sm.ndim == 2:
            sm = sm[:, :, None]
        if sm.ndim != 3 or sm.shape[1:] != (self.T, self.nd):
            raise ValueError(f"samples must be [n, {self.T}, {self.nd}]")
        vals = np.empty(sm.shape[0])
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_reached_simulate(self.h, st.ctypes.data_as(dp), sm.ctypes.data_as(dp), sm.shape[0],
                                                   float(discount), vals.ctypes.data_as(dp)))
        return vals

    def opt_table(self):
        """[rows, ndim + 3]: (t, state..., a1, a2) of every reached state in memo-map order."""
        n = C.c_size_t(0)
        self._check(self.lib.sdpb_reached_opt_table(self.h, None, C.byref(n)))
        rows = np.empty((n.value, self.ndim + 3))
        self._check(self.lib.sdpb_reached_opt_table(self.h, rows.ctypes.data_as(C.POINTER(C.c_double)), C.byref(n)))
        return rows

    def n_states(self):
        """Reached states of each period (T entries)."""
        out = (C.c_int64 * self.T)()
        self._check(self.lib.sdpb_reached_states(self.h, out))
        return list(out)

    def stats(self):
        s = A.SdpbStats()
        self._check(self.lib.sdpb_reached_stats(self.h, C.byref(s)))
        return {"evals": s.evals, "evals_executed": s.evals_executed, "solve_ms": s.solve_ms, "kernel_ms": s.kernel_ms,
                "launches": s.launches}


class Group:
    """`n` shards of one model on the given CUDA devices of THIS process (sdpb_group_*): the grid is cut into
    contiguous blocks, every shard holds only the window of V_t it reads, and rows travel between the shards' tables
    through peer-mapped device memory inside the library.  An ordinal may repeat (shards sharing one GPU)."""

    def __init__(self, spec: ModelSpec, devices, kernel: int = A.KERNEL_AUTO, dedup: bool = False, allow: int = 0,
                 profile: bool = False):
        self.lib = A.load()
        self.spec = spec
        self._model = spec.to_struct()
        opt = make_options(kernel=kernel, dedup=dedup, allow=allow | spec.allow, profile=profile)
        dev = (C.c_int32 * len(devices))(*devices)
        g = C.c_void_p()
        rc = self.lib.sdpb_group_create(C.byref(self._model), C.byref(opt), dev, len(devices), C.byref(g))
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_group_last_error(None).decode())
        self.g = g
        self.n = len(devices)
        self.shards = []
        for r in range(self.n):
            s = Solver.__new__(Solver)
            s.lib, s.spec, s._model = self.lib, spec, self._model
            s.h = C.c_void_p(self.lib.sdpb_group_shard(self.g, r))
            gi = A.SdpbGrid()
            s._check(self.lib.sdpb_grid_info(s.h, C.byref(gi)))
            s.grid, s.ndim, s.n_states, s.T = gi, gi.ndim, gi.n_states, gi.T
            s.close = lambda: None  # owned by the group
            self.shards.append(s)
        self.n_states, self.T, self.ndim = self.shards[0].n_states, self.shards[0].T, self.shards[0].ndim

    def _check(self, rc):
        if rc != A.SDPB_OK:
            raise A.SdpbError(rc, self.lib.sdpb_group_last_error(self.g).decode())

    def solve(self):
        self._check(self.lib.sdpb_group_solve(self.g))
        return self

    def value(self, period, states):
        st = np.ascontiguousarray(np.atleast_2d(np.asarray(states, dtype=np.float64)))
        n = st.shape[0]
        v, q = np.empty(n), np.empty(n)
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_group_value(self.g, period, st.ctypes.data_as(dp), n, v.ctypes.data_as(dp),
                                              q.ctypes.data_as(dp)))
        return v, q

    def period_tables(self, period):
        V, Q = np.empty(self.n_states), np.empty(self.n_states)
        dp = C.POINTER(C.c_double)
        self._check(self.lib.sdpb_group_period_tables(self.g, period, V.ctypes.data_as(dp), Q.ctypes.data_as(dp)))
        return V, Q

    def stats(self):
        s = A.SdpbStats()
        self._check(self.lib.sdpb_group_stats(self.g, C.byref(s)))
        return {"evals": s.evals, "solve_ms": s.solve_ms, "launches": s.launches, "kernel_used": s.kernel_used,
                "fp64_ops": s.fp64_ops, "evals_executed": s.evals_executed, "exchange_ms": s.exchange_ms}

    def close(self):
        if getattr(self, "g", None):
            self.lib.sdpb_group_destroy(self.g)
            self.g = None
            for s in self.shards:
                s.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
