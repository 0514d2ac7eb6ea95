"""The reached-state handle (sdpb_reached_*) on the two recorded T = 3 instances of the reference's two-product model
(MultiProductLeadtime.java:35-39 and 45-50), on one GPU, in one process.

    python tools/time_reached.py --parent-lib PATH [--reps 5] [--paths 10000]

PATH is a libsdpb200.so built from an earlier commit.  It is loaded beside this tree's library, and the two
sdpb_reached_solve calls are alternated `reps` times on each instance.  Reported: the device time (solve_ms) and host
wall time of each, as median and min..max, and whether the two give the same value, actions and state counts.  Then,
on this tree's library: sdpb_reached_open from the root, the device memory the open handle holds (the drop in free
device memory), a value query over every period-3 state, and a roll-out of `paths` paths from the root with demand
pairs drawn from the pmf support (fixed seed).  The first line names the GPU, its power limit and its maximum SM
clock.  One JSON line per measurement."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sdpb200 as S  # noqa: E402

INSTANCES = {  # (vals1, vals2), (probs1, probs2), the value the reference's author recorded
    "T3-4pairs": (([10, 30], [5, 15]), ([0.5, 0.5], [0.5, 0.5]), -76.56),
    "T3-9pairs": (([20, 30, 40], [10, 15, 20]), ([0.25, 0.5, 0.25], [0.25, 0.5, 0.25]), 91.19499999999998),
}


def pmf(vals, probs, T=3):
    rows = np.array([(a, b, pa * pb) for a, pa in zip(vals[0], probs[0]) for b, pb in zip(vals[1], probs[1])])
    return [rows.copy() for _ in range(T)]


def solve(lib, model, root):
    v, a1, a2, ms = C.c_double(), C.c_double(), C.c_double(), C.c_double()
    ns = (C.c_int64 * 3)()
    dp = C.POINTER(C.c_double)
    t0 = time.perf_counter()
    rc = lib.sdpb_reached_solve(C.byref(model), 0, root.ctypes.data_as(dp), C.byref(v), C.byref(a1), C.byref(a2), ns,
                                C.byref(ms))
    wall = (time.perf_counter() - t0) * 1e3
    if rc != 0:
        raise RuntimeError(f"sdpb_reached_solve: {rc}")
    return (v.value, a1.value, a2.value, list(ns)), ms.value, wall


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--paths", type=int, default=10000)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print(json.dumps({"gpu": gpu}), flush=True)
    new = S.abi.load()
    old = C.CDLL(os.path.abspath(args.parent_lib))
    old.sdpb_reached_solve.argtypes = new.sdpb_reached_solve.argtypes
    root = np.zeros(5)
    for name, (vals, probs, recorded) in INSTANCES.items():
        rec = S.CashRecursionMultiLead(pmf(vals, probs), Qbound=50)
        m = rec._m
        solve(new, m, root)  # warm-up: module load, pool
        solve(old, m, root)
        res = {"parent": ([], [], None), "this": ([], [], None)}
        for _ in range(args.reps):
            for key, lib in (("parent", old), ("this", new)):
                out, ms, wall = solve(lib, m, root)
                res[key][0].append(ms)
                res[key][1].append(wall)
                res[key] = (res[key][0], res[key][1], out)
        print(json.dumps({"instance": name, "what": "sdpb_reached_solve, alternated", "reps": args.reps,
                          "parent_solve_ms": summary(res["parent"][0]), "this_solve_ms": summary(res["this"][0]),
                          "parent_wall_ms": summary(res["parent"][1]), "this_wall_ms": summary(res["this"][1]),
                          "same_outputs": res["parent"][2] == res["this"][2], "value": res["this"][2][0],
                          "recorded": recorded, "n_states": res["this"][2][3]}), flush=True)

        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info(0)[0]
        t0 = time.perf_counter()
        rh = S.Reached(m, [root], device=0)
        open_wall = (time.perf_counter() - t0) * 1e3
        held = free0 - torch.cuda.mem_get_info(0)[0]
        st = rh.stats()
        rows = rh.opt_table()
        p3 = np.ascontiguousarray(rows[rows[:, 0] == 3, 1:6])
        t0 = time.perf_counter()
        v3, _, _ = rh.value(3, p3)
        query_wall = (time.perf_counter() - t0) * 1e3
        rng = np.random.default_rng(20261020)
        table = pmf(vals, probs)[0]
        samples = table[rng.choice(len(table), size=(args.paths, 3), p=table[:, 2])][:, :, :2]
        n0 = rh.n_states()
        t0 = time.perf_counter()
        paths = rh.simulate(root, samples)
        sim_wall = (time.perf_counter() - t0) * 1e3
        sim = rh.stats()
        print(json.dumps({"instance": name, "open_wall_ms": open_wall, "open_solve_ms": st["solve_ms"],
                          "open_kernel_ms": st["kernel_ms"], "evals": st["evals"], "device_bytes_held": held,
                          "bytes_per_state": held / sum(n0), "period3_states": len(p3), "query_wall_ms": query_wall,
                          "query_finite": bool(np.isfinite(v3).all()), "paths": args.paths,
                          "rollout_wall_ms": sim_wall, "rollout_kernel_ms": sim["kernel_ms"], "rounds": sim["launches"],
                          "states_added": sum(rh.n_states()) - sum(n0), "mean_path_value": float(paths.mean())}),
              flush=True)
        rh.close()


if __name__ == "__main__":
    main()
