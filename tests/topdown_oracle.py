"""ctypes access to the CPU references of sdpb_topdown_extend / sdpb_topdown_simulate (tests/topdown_oracle.cpp, which
includes the oracle unchanged).  Test infrastructure only.  The library is compiled on first use into a temporary
directory, keyed by a hash of its sources, so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_lib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "topdown_oracle.cpp"), os.path.join(ROOT, "oracle", "sdp_oracle.cpp"),
           os.path.join(ROOT, "include", "sdpb200.h")]
# the oracle's own flags (oracle/Makefile): Java never fuses multiply-add, so neither may the reference
CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-Wall", "-Wextra",
            "-shared"]

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
    out_dir = os.path.join(tempfile.gettempdir(), "sdpb200-topdown-oracle")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libtopdown_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["g++", *CXXFLAGS, "-o", tmp, SOURCES[0]], check=True, capture_output=True)
        os.replace(tmp, so)
    lib = C.CDLL(so)
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    lib.oracle_topdown_at.argtypes = [vp, C.POINTER(C.c_int), dp, C.c_int, dp, C.c_int64, dp, dp]
    lib.oracle_topdown_at.restype = C.c_int64
    lib.oracle_topdown_simulate.argtypes = [vp, dp, dp, C.c_int, C.c_double, dp, dp, C.c_int64, dp]
    lib.oracle_topdown_simulate.restype = C.c_int64
    _lib = lib
    return lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def topdown_at(spec, periods, states):
    """getExpectedValue on states of any period, in call order, on one memo -> (rows [n, ndim+3] = [t, state..., Q, V]
    in memo order, the calls' values, evals)"""
    lib = load()
    m = spec.to_struct()
    st = np.ascontiguousarray(np.atleast_2d(np.asarray(states, dtype=np.float64)))
    pr = np.ascontiguousarray(periods, dtype=np.int32)
    assert len(pr) == st.shape[0]
    _, nd = oracle_lib.grid(spec)
    iv = np.empty(st.shape[0])
    ev = C.c_double()
    ip = pr.ctypes.data_as(C.POINTER(C.c_int))
    n = lib.oracle_topdown_at(C.byref(m), ip, _dp(st), st.shape[0], None, 0, _dp(iv), C.byref(ev))
    rows = np.empty((n, nd + 3))
    lib.oracle_topdown_at(C.byref(m), ip, _dp(st), st.shape[0], _dp(rows), n, _dp(iv), C.byref(ev))
    return rows, iv, ev.value


def topdown_simulate(spec, init_state, samples, discount=1.0):
    """Simulation.java:59-70 over one memoised recursion -> (per-path sums, memo rows afterwards as topdown_at, evals)"""
    lib = load()
    m = spec.to_struct()
    st = np.ascontiguousarray(init_state, dtype=np.float64)
    sm = np.ascontiguousarray(samples, dtype=np.float64)
    _, nd = oracle_lib.grid(spec)
    vals = np.empty(sm.shape[0])
    ev = C.c_double()
    cap = 4096
    while True:
        rows = np.empty((cap, nd + 3))
        n = lib.oracle_topdown_simulate(C.byref(m), _dp(st), _dp(sm), sm.shape[0], float(discount), _dp(vals),
                                        _dp(rows), cap, C.byref(ev))
        if n <= cap:
            return vals, rows[:n], ev.value
        cap = n
