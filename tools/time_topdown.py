"""The reached-state engine (sdpb_topdown_*) on one B200: reached states per period, evaluations, solve / backward-kernel
time and evaluations/s, beside the dense solve of the same grid and the one-thread rate of the reference's memoised
recursion (bench.py's oracle_topdown figure).

    python tools/time_topdown.py [c1] [c4] [c3]     # default: all three; one JSON line per configuration

C1 from x = 0, C4 (lead time 2, T = 20) from (0, 0, 0), C3 (cash, T = 12) from (0, 100).  The dense time is the second
of two sdpb_solve calls; the top-down time is one sdpb_topdown_solve (forward + backward), measured with CUDA events
inside the library.  Neither overwrites the L2 between runs."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import sdpb200 as S  # noqa: E402
import bench  # noqa: E402

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
print(json.dumps({"gpu": gpu}), flush=True)
for name in sys.argv[1:] or ["c1", "c4", "c3"]:
    spec = {"c1": S.configs.c1, "c3": S.configs.c3, "c4": S.configs.c4}[name]()
    init = bench.INIT[name]
    t0 = time.perf_counter()
    td = S.TopDown(spec, init, device=0)
    wall = time.perf_counter() - t0
    st = td.stats()
    states = td.n_states()
    v_td = td.value(1, init)[0][0]
    td.close()
    dense = S.Solver(spec, device=0)
    dense.solve()
    dense.solve()
    ds = dense.stats()
    v_dense = dense.value(1, init)[0][0]
    dense.close()
    rate = bench.time_topdown(S, name, spec)[0]
    print(json.dumps({
        "config": name, "init": init[0], "value_equal_to_dense": bool(v_td == v_dense),
        "topdown": {"states_per_period": states, "evals": st["evals"], "solve_ms": st["solve_ms"],
                    "backward_kernel_ms": st["kernel_ms"], "evals_per_s": st["evals"] / (st["solve_ms"] * 1e-3),
                    "wall_s": wall},
        "dense": {"grid_states": dense.n_states, "evals": ds["evals"], "solve_ms": ds["solve_ms"],
                  "evals_per_s": ds["evals"] / (ds["solve_ms"] * 1e-3)},
        "oracle_topdown_1thread_evals_per_s": rate}), flush=True)
