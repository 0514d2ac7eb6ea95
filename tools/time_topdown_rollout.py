"""The top-down engine's policy roll-out (sdpb_topdown_simulate) on one B200, beside the dense roll-out (sdpb_simulate).

    python tools/time_topdown_rollout.py [c1] [c2]     # default: both; one JSON line per configuration

Each configuration runs 10,000 Latin-hypercube paths (generate_lh_samples, fixed seed) from x = 0: the reference
drivers' Simulation step.  A top-down handle is solved from x = 0, then rolled out; LHS strata beyond the pmf's
truncation quantile reach states the solve did not visit, which the roll-out solves as it meets them.  Reported: the
solve time, the roll-out time (host wall time of the call, and the roll-out kernels' device time), the rounds, the
states and evaluations the roll-out added, and on the same samples the dense sdpb_simulate time (the second of two
calls, after a dense solve) and whether its per-path values are == the top-down ones.  The first line names the GPU,
its power limit and its maximum SM clock."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import sdpb200 as S  # noqa: E402

MEANS = {"c1": [20, 40, 60, 40], "c2": S.configs.C2_MEANS}
PATHS = 10000

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
print(json.dumps({"gpu": gpu}), flush=True)
for name in sys.argv[1:] or ["c1", "c2"]:
    spec = {"c1": S.configs.c1, "c2": S.configs.c2}[name]()
    samples = S.generate_lh_samples([S.PoissonDist(m) for m in MEANS[name]], PATHS)
    init = [0.0]
    td = S.TopDown(spec, [init], device=0)
    solve = td.stats()
    n0 = td.n_states()
    t0 = time.perf_counter()
    v_td = td.simulate(init, samples)
    wall = time.perf_counter() - t0
    sim = td.stats()
    n1 = td.n_states()
    td.close()
    dense = S.Solver(spec, device=0).solve()
    dense.simulate(init, samples)
    t0 = time.perf_counter()
    v_dense = dense.simulate(init, samples)
    dense_ms = (time.perf_counter() - t0) * 1e3
    dense.close()
    print(json.dumps({
        "config": name, "paths": PATHS, "init": init,
        "solve_ms": solve["solve_ms"], "solve_states_per_period": n0, "solve_evals": solve["evals"],
        "rollout_ms": wall * 1e3, "rollout_lib_ms": sim["solve_ms"], "rollout_kernel_ms": sim["kernel_ms"],
        "rounds": sim["launches"], "states_added_per_period": [b - a for a, b in zip(n0, n1)],
        "evals_added": sim["evals"] - solve["evals"], "mean": float(v_td.mean()),
        "dense_simulate_ms": dense_ms, "per_path_equal_to_dense": bool(np.array_equal(v_td, v_dense))}), flush=True)
