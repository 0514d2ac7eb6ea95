"""ctypes access to the CPU references of the reached-state handle (tests/reached_oracle.cpp, which includes the oracle
unchanged).  Test infrastructure only.  The library is compiled on first use into a temporary directory, keyed by a
hash of its sources, so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "reached_oracle.cpp"), os.path.join(ROOT, "oracle", "sdp_oracle.cpp"),
           os.path.join(ROOT, "include", "sdpb200.h")]
# the oracle's own flags (oracle/Makefile): Java never fuses multiply-add, so neither may the reference
CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-Wall", "-Wextra",
            "-shared"]
NDIM = {0: 5, 1: 3, 2: 3, 3: 2}

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256()
    for p in SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(CXXFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), "sdpb200-reached-oracle")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libreached_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["g++", *CXXFLAGS, "-o", tmp, SOURCES[0]], check=True, capture_output=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    lib.oracle_reached_at.argtypes = [vp, C.POINTER(C.c_int), dp, C.c_int, dp, C.c_int64, dp, dp]
    lib.oracle_reached_at.restype = C.c_int64
    lib.oracle_reached_simulate.argtypes = [vp, dp, dp, C.c_int, C.c_double, dp, dp, C.c_int64, dp]
    lib.oracle_reached_simulate.restype = C.c_int64
    _lib = lib
    return lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def reached_at(model, periods, states):
    """getExpectedValue on states of any period, in call order, on one memo of the `SdpbReachedModel` -> (rows
    [n, ndim + 4] = [t, state..., a1, a2, V] in memo-map order, the calls' values, evals)"""
    lib = load()
    nd = NDIM[model.kind]
    st = np.ascontiguousarray(np.asarray(states, dtype=np.float64).reshape(-1, nd))
    pr = np.ascontiguousarray(periods, dtype=np.int32)
    assert len(pr) == st.shape[0]
    vals, ev = np.empty(st.shape[0]), C.c_double()
    ip = pr.ctypes.data_as(C.POINTER(C.c_int))
    n = lib.oracle_reached_at(C.byref(model), ip, _dp(st), st.shape[0], None, 0, _dp(vals), C.byref(ev))
    assert n >= 0, "kind 0 needs one demand table for every period"
    rows = np.empty((n, nd + 4))
    lib.oracle_reached_at(C.byref(model), ip, _dp(st), st.shape[0], _dp(rows), n, _dp(vals), C.byref(ev))
    return rows, vals, ev.value


def reached_simulate(model, init_state, samples, discount=1.0):
    """The roll-out loop over one memo -> (per-path values, memo rows afterwards as reached_at, evals).  `samples`:
    [n, T, 2] for two products, [n, T] (or [n, T, 1]) for one."""
    lib = load()
    nd = NDIM[model.kind]
    st = np.ascontiguousarray(init_state, dtype=np.float64)
    sm = np.ascontiguousarray(samples, dtype=np.float64)
    vals, ev = np.empty(sm.shape[0]), C.c_double()
    n = lib.oracle_reached_simulate(C.byref(model), _dp(st), _dp(sm), sm.shape[0], float(discount), _dp(vals), None, 0,
                                    C.byref(ev))
    assert n >= 0, "kind 0 needs one demand table for every period"
    rows = np.empty((n, nd + 4))
    lib.oracle_reached_simulate(C.byref(model), _dp(st), _dp(sm), sm.shape[0], float(discount), _dp(vals), _dp(rows), n,
                                C.byref(ev))
    return vals, rows, ev.value
