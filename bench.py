#!/usr/bin/env python
"""bench.py — SDP solve time and state-action-demand evaluations/s (fp64) on N B200s.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W  # CPU arm: the oracle port on host cores

A "step" is one full-horizon solve (T backward-induction periods) of the workload.  The default
workload is BASELINE.json configs[3], the instance north_star partitions across GPUs: src/leadtime
with lead time 2, (x, q1, q2) state, 10,211,201 states x 101 actions x 25 demand points, T = 20, on a FIXED
grid (strong scaling: at N GPUs the grid is cut into N bands of inventory rows, every rank holds only
the window of V_t it reads, and after each period the ranks copy the rows their neighbours read
straight into the neighbours' tables through peer-mapped memory inside libsdpb200 -- no collective
library on the data path).  The other configs (C1, C2, C3, the C5 sweep) are solved once each and
reported under "configs".

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

REF_F = {"c1": 20, "c2": 20, "c3": 41, "c4": 20, "c5": 20}  # SURVEY.md section 8(d): fp64 ops per evaluation as written
KERNEL_NAMES = {1: "bi_generic", 2: "bi_inv_tiled", 3: "bi_backorder_staged", 4: "bi_cash_int", 5: "bi_inv_tiled2",
                6: "bi_lead_slab", 7: "bi_lead_col", 8: "bi_cash_diag", 9: "bi_lead_q2", 14: "bi_lead_q2m", 15: "collapsed_levels + collapsed_actions", 10: "bi_two_product_row",
                11: "bi_inv_fused", 12: "bi_cash_row", 13: "bi_cash_tail"}
METRIC = "state-action-demand evaluations/s (fp64), full-horizon SDP solve"
UNIT = "evals/s"
INIT = {"c1": [[0.0]], "c2": [[0.0]], "c3": [[0.0, 100.0]], "c4": [[0.0, 0.0, 0.0]], "c5": [[0.0]]}
GOLDEN_KEY = {"c3": "c3", "c4": "c4"}  # tests/golden/fullsize.json entries (c5 only at 1e7 states)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: the library's own peer exchange (default) or the round-1 torch.distributed path")
    ap.add_argument("--states-per-gpu", type=int, default=10_000_000, help="C5 only (weak scaling)")
    ap.add_argument("--kernel", default="auto", choices=["auto", "generic", "tiled", "tiled2"])
    ap.add_argument("--dedup", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the one-shot solves of the other configurations")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="one GPU: write the timed solve's value and policy tables to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU solve's tables; the reference arm solves a sub-grid only")
    return args


def make_spec(S, name, n_gpus, states_per_gpu):
    c = S.configs
    if name == "c5":
        return c.c5(n_states=states_per_gpu * n_gpus)
    return {"c1": c.c1, "c2": c.c2, "c3": c.c3, "c4": c.c4}[name]()


def workload_desc(spec, name, n_gpus, exchange="p2p"):
    D = [len(r) for r in spec.pmf]
    part = "none"
    if n_gpus > 1:
        part = (f"state grid in {n_gpus} contiguous blocks (bands of inventory rows); every rank holds the window of "
                "V_t its kernels read; per period ")
        part += ("each rank copies the rows its peers read into their tables through CUDA-IPC peer-mapped memory and "
                 "raises a device-side flag (libsdpb200: sdpb_peer_attach), no collective library"
                 if exchange == "p2p" else "torch.distributed point-to-point halo exchange / all-gather over NCCL")
    return {
        "workload": {
            "c1": "C1 src/sdp single-item lot sizing T=4 Poisson[20,40,60,40] 1001 states x 501 actions",
            "c2": "C2 src/capacitated T=20 2001 states x 101 actions",
            "c3": "C3 src/cash (inventory, cash) 1,002,501 states x <=201 actions x 200 demands T=12",
            "c4": "C4 src/leadtime L=2 10,211,201 states x 101 actions x 25 demands T=20",
            "c5": f"C5 synthetic sweep family A: {spec.n_states()} states x {spec.max_order_idx + 1} actions x "
                  f"{D[0]} demand points, T={spec.T}",
        }[name],
        "T": spec.T, "demand_points": D[0] if len(set(D)) == 1 else D,
        "actions": spec.max_order_idx + 1,
        "partition": part,
        "l2": "inputs larger than L2: a C4 step writes 12 B x 10.2e6 states x 20 periods = 2.45 GB of tables (126 MB L2), "
              "and its first launch (period T) reads no table at all, so nothing cached by the previous timed step "
              "can be reused; within a step V_{t+1} is what the previous period left behind, as in any solve",
    }


# ---- clocks ---------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v == "Active":
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU arm ----------------------------------------------------------------------------------
def java_probe():
    """Is there a JVM on this box?  (BASELINE.md: time the reference Java itself when one is found.)"""
    out = {}
    for exe in ("java", "javac"):
        try:
            r = subprocess.run([exe, "-version"], capture_output=True, text=True, timeout=20)
            out[exe] = (r.stderr or r.stdout).strip().splitlines()[0] if r.returncode == 0 else f"exit {r.returncode}"
        except FileNotFoundError:
            out[exe] = "not found"
        except Exception as e:  # noqa: BLE001
            out[exe] = f"error: {e}"
    out["usable"] = all(v != "not found" and not v.startswith(("exit", "error")) for v in (out["java"], out["javac"]))
    return out


def cpu_sample_spec(S, name, spec, rows):
    """The same model on a sub-grid of `rows` inventory levels: same actions, demand table, horizon, cash axis and
    pipeline axes -- the per-state work of the CPU solve does not depend on how many inventory rows there are."""
    c = S.configs
    if name == "c3":
        return c.c3(inv_max=max(1, rows - 1))
    if name == "c4":
        return c.c4(inv_half=max(1, rows // 2))
    import copy
    s = copy.copy(spec)
    half = rows // 2
    s.inv_min, s.inv_max = float(-half), float(rows - half - 1)
    return s


def states_per_row(name):
    return {"c3": 2001, "c4": 101 * 101}.get(name, 1)


def time_dense(sample, threads=0):
    import oracle_lib as O
    t0 = time.perf_counter()
    _, _, ev, _ = O.dense(sample, threads)
    return ev, time.perf_counter() - t0


def calibrate_rows(S, name, spec, seconds, threads=0):
    """Rows of the sub-grid that take about `seconds` of oracle_dense on this box's host cores."""
    import oracle_lib as O
    small = cpu_sample_spec(S, name, spec, {"c3": 2, "c4": 3}.get(name, 256))
    ev, dt = time_dense(small, threads)
    rows_small = O.grid(small)[0] // states_per_row(name)
    rate = ev / max(dt, 1e-3)
    per_row = ev / rows_small
    full_rows = O.grid(spec)[0] // states_per_row(name)
    return int(max(rows_small, min(full_rows, rate * seconds / per_row)))


def time_topdown(S, name, spec):
    """The reference's own control flow (memoised top-down recursion, one thread) from the initial state, on an
    instance cut down until it takes seconds: the first 3 periods of C3 / C4 on a few inventory rows, a 2048-state
    grid for the 1-D families.  A rate (evaluations/s of the literal recursion), not a solve of the workload."""
    import oracle_lib as O
    c = S.configs
    if name == "c3":
        sample = c.c3(T=3, inv_max=7)
    elif name == "c4":
        sample = c.c4(T=3, inv_half=3)
    else:
        sample = cpu_sample_spec(S, name, spec, 2048)
    t0 = time.perf_counter()
    vis, _, ev = O.topdown(sample, INIT[name])
    dt = time.perf_counter() - t0
    return ev / dt, ev, dt, len(vis), O.grid(sample)[0]


def workload_evals(name, spec):
    return 4.612e11 if name == "c3" else spec.evals_dense()  # (C3's action sets depend on the cash level)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle_lib as O
    import sdpb200 as S
    name = args.workload
    spec = make_spec(S, name, 1, args.states_per_gpu)
    cores = os.cpu_count() or 1
    # size one step to ~ (150 s budget) / (steps + warmup)
    per_step = max(2.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    rows = calibrate_rows(S, name, spec, per_step)
    sample = cpu_sample_spec(S, name, spec, rows)
    n_sample, n_full = O.grid(sample)[0], O.grid(spec)[0]
    for _ in range(max(0, args.warmup - 1)):
        time_dense(sample)
    t_total, ev_total = 0.0, 0.0
    for _ in range(args.steps):
        e, d = time_dense(sample)
        t_total += d
        ev_total += e
    value = ev_total / t_total
    td_rate, td_ev, td_dt, td_rows, td_states = time_topdown(S, name, spec)
    what = (f"oracle_dense (C++ restatement of the reference loop, {cores} host threads) on a {n_sample}-state sub-grid "
            f"({rows} of the inventory rows) of the {n_full}-state workload; all {spec.max_order_idx + 1} actions x "
            f"{len(spec.pmf[0])} demands x T={spec.T}")
    cfg = workload_desc(spec, name, 1)
    cfg["workload"] += f" -- CPU arm: RATE EXTRAPOLATED from a {n_sample}-state sub-grid (the full grid is not solved)"
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "ms_per_step_note": "time of one sub-grid solve, not of the workload; the full workload at this rate would take "
                            f"{workload_evals(name, spec) / value:.0f} s",
        "higher_is_better": True, "scaling": "strong" if name in ("c3", "c4") else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": what,
                         "java_probe": java_probe(),
                         "topdown_1thread": {"value": td_rate, "unit": UNIT,
                                             "sample": f"oracle_topdown (the reference's memoised recursion, 1 thread) from "
                                                       f"the initial state on a cut-down instance ({td_states} states per period, first periods "
                                                       f"only): {td_rows} visited states, {td_dt:.1f} s -- this is the work the "
                                                       "single-threaded Java does per evaluation"},
                         "note": "the reference is single-threaded Java; no JDK in the image (probe above), so the C++ port "
                                 "is timed: multi-threaded dense solve as `value`, the literal 1-thread recursion beside it"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))
    return 0


# ---- GPU arm ----------------------------------------------------------------------------------
def per_step_counts(sh, sync):
    """(evals, evals_executed, fp64_ops, kernel, launches) of ONE step (the library resets its counters per solve)."""
    sh.step()
    sync()
    if sh.world > 1 and sh.exchange_kind != "p2p":  # stepped period by period: the counters accumulate
        a = sh.solver.stats()
        sh.step()
        sync()
        b = sh.solver.stats()
        return (b["evals"] - a["evals"], b["evals_executed"] - a["evals_executed"], b["fp64_ops"] - a["fp64_ops"],
                b["kernel_used"], b["launches"] - a["launches"])
    b = sh.solver.stats()
    return b["evals"], b["evals_executed"], b["fp64_ops"], b["kernel_used"], b["launches"]


def table_hash_check(solver, gold):
    """Whole grid, every period: SHA-256 of V_t / Q_t bytes against the frozen whole-grid oracle run."""
    import numpy as np
    V, Q = np.empty(solver.n_states), np.empty(solver.n_states)
    for t in range(1, solver.T + 1):
        solver.period_tables(t, out_v=V, out_q=Q)
        if hashlib.sha256(V.tobytes()).hexdigest() != gold["sha256_V"][t - 1]:
            return False
        if hashlib.sha256(Q.tobytes()).hexdigest() != gold["sha256_Q"][t - 1]:
            return False
    return True


def sample_check(spec, solver, n=32, seed=5):
    """Inductive check on a sample: recompute V_t, Q_t on the CPU (the oracle, as the checker) at random states from
    the GPU's own V_{t+1}, every period."""
    import numpy as np
    import oracle_lib as O
    rng = np.random.default_rng(seed)
    idx = np.unique(np.concatenate([[0, solver.n_states - 1], rng.integers(0, solver.n_states, n)]))
    Vn = None
    V, Q = np.empty(solver.n_states), np.empty(solver.n_states)
    for t in range(spec.T, 0, -1):
        solver.period_tables(t, out_v=V, out_q=Q)
        vo, qo = O.step_states(spec, t, Vn, idx)
        if not (np.array_equal(V[idx], vo) and np.array_equal(Q[idx], qo)):
            return False
        Vn = V.copy()
    return True


DUMP_BYTES = 56 << 20  # V, Q and the state index together: the whole dump stays under 64 MB


def dump_outputs(out_dir, solver, init, seed=0):
    """What a caller of the timed solve receives, as float64 .npy files, for comparing two builds output for output:
    V.npy / Q.npy [T, k]: the value and order-quantity tables of every period (sdpb_period_tables) at the k flattened
    state indices in state_index.npy -- every state when that fits in DUMP_BYTES, else a fixed sample drawn with
    `seed` (the same states in every run of the same workload); V1_init.npy / Q1_init.npy: sdpb_value at the
    workload's initial state."""
    import numpy as np
    n, T = solver.n_states, solver.T
    k = min(n, DUMP_BYTES // (16 * T + 8))
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))
    V, Q = np.empty((T, k)), np.empty((T, k))
    Vt, Qt = np.empty(n), np.empty(n)
    for t in range(1, T + 1):
        solver.period_tables(t, out_v=Vt, out_q=Qt)
        V[t - 1], Q[t - 1] = Vt[idx], Qt[idx]
    v1, q1 = solver.value(1, init)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("V", V), ("Q", Q), ("state_index", idx.astype(np.float64)), ("V1_init", v1), ("Q1_init", q1)):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def verify_vs_unsharded(S, torch, dist, sp, sharded, local, dedup):
    """Multi-GPU result check (outside every timed region): each rank re-solves the WHOLE grid by itself and compares
    its own block of V_1 and Q_1, bit for bit, with what the sharded solve (real peer exchange) left in its tables."""
    import numpy as np
    torch.cuda.synchronize()
    sharded.solver.sync()
    Vm, Qm = sharded.solver.shard_tables(1)
    lo_, hi_ = sharded.lo, sharded.hi
    with S.Solver(sp, device=local, dedup=dedup) as ref:
        ref.solve()
        Vr, Qr = ref.period_tables(1)
    ok = bool(np.array_equal(Vm, Vr[lo_:hi_]) and np.array_equal(Qm, Qr[lo_:hi_]))
    okt = torch.tensor([1 if ok else 0], dtype=torch.int32, device=f"cuda:{local}")
    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    return bool(int(okt[0]))


def next_rows(S, device):
    """SURVEY.md section 8 'next' rows, one timed invocation each (wall clock around the blocking C-ABI
    calls; second call timed so one-off allocations are outside)."""
    import numpy as np
    res = {}

    def timed(fn, reps=2):
        for _ in range(reps - 1):
            fn()
        t0 = time.perf_counter()
        r = fn()
        return r, time.perf_counter() - t0

    sp = S.configs.c1()
    with S.Solver(sp, device=device) as s:
        s.solve()
        _, dt_r = timed(lambda: s.reach([[0.0]]))
        tab, dt_t = timed(lambda: s.opt_table())
        res["f1_opt_table_c1"] = {"reach_ms": dt_r * 1e3, "opt_table_ms": dt_t * 1e3, "rows": int(len(tab)),
                                  "what": "sdpb_reach from x0 = 0 + sdpb_opt_table (Recursion.getOptTable())"}
        rng = np.random.default_rng(7)
        n = 200_000
        samples = np.stack([rng.choice(r[:, 0], size=n, p=r[:, 1] / r[:, 1].sum()) for r in sp.pmf], axis=1)
        vals, dt_s = timed(lambda: s.simulate([0.0], samples))
        v1, _ = s.value(1, [[0.0]])
        res["f2_simulate_c1"] = {"paths": n, "ms": dt_s * 1e3, "paths_per_s": n / dt_s, "mean": float(vals.mean()),
                                 "V1_init": float(v1[0]),
                                 "what": "sdpb_simulate, host samples in / per-path sums out (Simulation.java:53-74)"}
    d1, d2 = S.PoissonDist(5), S.PoissonDist(6)
    rows = S.GetPmfMulti([[d1] * 3, [d2] * 3], 0.999, 1).tables()
    sp = S.two_product_cash_model(rows, price=(4.0, 5.0), vari_cost=(2.0, 3.0), salvage=(1.0, 1.0), q_bound=20,
                                  inv_max=40.0, cash_min=0.0, cash_max=400.0)
    with S.Solver(sp, device=device) as s:
        s.solve()
        _, dt = timed(lambda: s.solve(), reps=1)
        st = s.stats()
        res["f3_two_product"] = {"states": int(s.n_states), "T": sp.T, "demand_pairs": int(len(rows[0])),
                                 "solve_ms": dt * 1e3, "evals": st["evals"], "evals_per_s": st["evals"] / dt,
                                 "kernel": KERNEL_NAMES.get(st["kernel_used"]),
                                 "what": "CashRecursionMulti + MultiItemCash.java:69-121 lambdas, 41 x 41 x 401 grid, "
                                         "Qbound 20 (the reference's 201 x 201 x 10001 dense grid is 4e8 states)"}
    # f-3, the reference's scaling wall: two products + lead time + un-quantised cash, solved over the reached states
    import numpy as np
    rows = np.array([(a, b, pa * pb) for a, pa in zip([10, 30], [0.5, 0.5]) for b, pb in zip([5, 15], [0.5, 0.5])], dtype=float)
    rec = S.CashRecursionMultiLead([rows.copy() for _ in range(3)], Qbound=50, device=device)
    t0 = time.perf_counter()
    val = rec.getExpectedValue(S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0))
    dt = time.perf_counter() - t0
    act = rec.getAction(S.CashStateMultiLead(1, 0, 0, 0, 0, 0.0))
    ev = float(sum(rec.n_states)) * 2500 * 4
    res["f3_multilead_T3"] = {"states_per_period": [int(x) for x in rec.n_states], "evals": ev, "device_ms": rec.solve_ms,
                              "wall_ms": dt * 1e3, "evals_per_s": ev / (rec.solve_ms * 1e-3), "value": val,
                              "Q1": act.getFirstAction(), "Q2": act.getSecondAction(),
                              "reference_record": "final optimal cash is -76.56, Q1 = 30, Q2 = 15, running time is 1568.0s "
                                                  "(src/cash/overdraft/MultiProductLeadtime.java:45-50)",
                              "matches_reference_record": bool(val == -76.56 and act.getFirstAction() == 30 and act.getSecondAction() == 15),
                              "what": "CashRecursionMultiLead + MultiProductLeadtime.java:150-224 lambdas through sdpb_reached_solve: "
                                      "forward enumeration of the reached states (expand, sort, unique), backward induction with "
                                      "binary-search successor lookup"}
    sp = S.workforce_model([0.5, 0.5, 0.5])
    with S.Solver(sp, device=device) as s:
        s.solve()
        _, dt = timed(lambda: s.solve(), reps=1)
        st = s.stats()
        v1, q1 = s.value(1, [[0.0]])
        res["f4_workforce"] = {"states": int(s.n_states), "T": sp.T, "solve_ms": dt * 1e3, "evals": st["evals"],
                               "evals_per_s": st["evals"] / dt, "kernel": "bi_staff", "V1_init": float(v1[0]),
                               "Q1_init": float(q1[0]),
                               "what": "StaffRecursion, WorkforcePlanning.java instance: 601 staff levels x 501 hires x "
                                       "Binomial(y, 0.5) turnover, T = 3"}
    return res


def run_gpu(args):
    import numpy as np
    import torch
    import sdpb200 as S

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libsdpb200 has no CPU path")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs --gpus 1: a shard holds only its block of the tables")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    par = S.package.parallel
    _CAI = par._CAI
    name = args.workload
    stream = torch.cuda.Stream(device=local)
    dev = f"cuda:{local}"

    def ShardedSolve(spec_, rank_, world_, kernel_, dedup_, profile=False):
        return par.ShardedSolve(S.Solver, torch, dist if world_ > 1 else None, spec_, rank_, world_, local, stream,
                                kernel_, dedup_, exchange=args.exchange, profile=profile)

    kernel = {"auto": S.KERNEL_AUTO, "generic": S.KERNEL_GENERIC, "tiled": S.KERNEL_TILED,
              "tiled2": S.KERNEL_TILED2}[args.kernel]
    spec = make_spec(S, name, world, args.states_per_gpu)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max_sum(vals):
        if world == 1:
            return list(vals), list(vals)
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        mx, sm = t.clone(), t.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        return [float(x) for x in mx], [float(x) for x in sm]

    with torch.cuda.stream(stream):
        sh = ShardedSolve(spec, rank, world, kernel, args.dedup)
        for _ in range(max(0, args.warmup - 1)):
            sh.step()
        barrier()
        ev_step, evx_step, fp_step, kernel_used, launches_step = per_step_counts(sh, barrier)  # the last warm-up step
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _ in range(args.steps):
            sh.step()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if rank == 0 else None
        (ms, _, _, _), (_, ev_total, fp_total, launches_total) = reduce_max_sum(
            [ms, ev_step * args.steps, fp_step * args.steps, launches_step * args.steps])
        value = ev_total / (ms * 1e-3)
        dev_bytes = sh.solver.grid.device_bytes
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, sh.solver, INIT[name])
        bytes_out, bytes_in = sh.bytes_out, sh.bytes_in

        # ---- verification of the timed workload's result (outside every timed region) ----
        verify = {}
        if not args.no_verify:
            if world == 1:
                verify["verified_vs_oracle_sample"] = bool(sample_check(spec, sh.solver))
                gold_path = os.path.join(ROOT, "tests", "golden", "fullsize.json")
                key = GOLDEN_KEY.get(name) or ("c5_1e7" if name == "c5" and spec.n_states() == 10_000_000 else None)
                if key and os.path.exists(gold_path) and not args.dedup:
                    gold = json.load(open(gold_path)).get(key)
                    if gold and np.array_equal(np.asarray(gold["pmf"][0]), np.asarray(spec.pmf[0])):
                        verify["verified_vs_golden_hash"] = bool(table_hash_check(sh.solver, gold))
                        verify["golden"] = f"tests/golden/fullsize.json[{key}]: whole grid, all {spec.T} periods, SHA-256"
            else:
                verify["verified_vs_unsharded"] = verify_vs_unsharded(S, torch, dist, spec, sh, local, args.dedup)

        # ---- per-period breakdown of the exchange (N > 1): two extra, profiled solves ----
        period_profile = None
        if world > 1 and args.exchange == "p2p":
            sp_ = ShardedSolve(spec, rank, world, kernel, args.dedup, profile=True)
            for _ in range(2):
                sp_.step()
                sp_.solver.sync()
            prof = torch.tensor(sp_.solver.period_profile(), dtype=torch.float64, device=dev)  # [T, 3]
            mx, mn = prof.clone(), prof.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(mn, op=dist.ReduceOp.MIN)
            period_profile = {
                "columns": ["kernels_ms", "push_and_flag_ms", "wait_for_peers_ms"],
                "rank0": [[round(float(x), 4) for x in row] for row in prof.cpu()],
                "max_over_ranks": [[round(float(x), 4) for x in row] for row in mx.cpu()],
                "min_over_ranks": [[round(float(x), 4) for x in row] for row in mn.cpu()],
                "sum_max_over_ranks_ms": [round(float(x), 3) for x in mx.sum(dim=0).cpu()],
                "what": "device time per period (period 1 first) of one solve, CUDA events on each rank's stream: the period's "
                        "kernels / peer copies + flag store / spin on the peers' flags (sdpb_period_profile)"}
            dist.barrier()
            sp_.close()

        # ---- e2e: through the C-ABI with host buffers; H2D of the descriptor tables and D2H of the
        # period-1 value/policy tables inside the timed region, every step ----
        e2e_steps = max(1, min(args.steps, 3))
        host_v = host_q = None  # the caller's result buffers: page-locked host memory, allocated once (warm-up cycle)
        d2h = h2d = 0
        phases = {"create_s": 0.0, "solve_s": 0.0, "fetch_s": 0.0, "destroy_s": 0.0}
        for e2e_it in range(e2e_steps + 1):  # iteration 0 is an untimed warm-up of the whole cycle
            if e2e_it <= 1:  # (re)start the clock after the warm-up cycle
                phases = {k: 0.0 for k in phases}
                barrier()
                t0 = time.perf_counter()
            p0 = time.perf_counter()
            s2 = ShardedSolve(spec, rank, world, kernel, args.dedup)
            p1 = time.perf_counter()
            s2.step()
            s2.solver.sync()
            p2 = time.perf_counter()
            nloc = s2.hi - s2.lo
            if world == 1:
                s2.solver.value(1, INIT[name])
                if host_v is None:
                    host_v = torch.empty(s2.solver.n_states, dtype=torch.float64).pin_memory().numpy()
                    host_q = torch.empty(s2.solver.n_states, dtype=torch.float64).pin_memory().numpy()
                s2.solver.period_tables(1, out_v=host_v, out_q=host_q)
                d2h = s2.n * 16 + 16
            else:
                dv, dq = s2.solver.device_tables(1)  # first elements held: V_1[window_lo], Q_1[shard_lo]
                wlo = s2.solver.grid.window_lo
                Vt = torch.as_tensor(_CAI(dv + 8 * (s2.lo - wlo), nloc, "<f8"), device=dev)
                Qt = torch.as_tensor(_CAI(dq, nloc, "<i4"), device=dev)
                if host_v is None:  # this rank's block of the result tables, page-locked
                    host_v = torch.empty(nloc, dtype=torch.float64).pin_memory()
                    host_q = torch.empty(nloc, dtype=torch.int32).pin_memory()
                host_v.copy_(Vt, non_blocking=True)
                host_q.copy_(Qt, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                d2h = nloc * 12
            npmf = sum(len(r) for r in spec.pmf)
            h2d = npmf * 28 + spec.T * 32
            p3 = time.perf_counter()
            if world > 1:
                dist.barrier()  # nobody unmaps a table while a peer may still be raising flags in it
            s2.close()
            p4 = time.perf_counter()
            for k, v in zip(phases, (p1 - p0, p2 - p1, p3 - p2, p4 - p3)):
                phases[k] += v / e2e_steps
        barrier()
        e2e_s = time.perf_counter() - t0
        (e2e_s,), _ = reduce_max_sum([e2e_s])
        e2e_value = (ev_total / args.steps) * e2e_steps / e2e_s

    out = None
    if rank == 0:
        peaks = S.abi.microbench(local)
        mp = {}
        try:
            mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        achieved = fp_total / (ms * 1e-3) / 1e12 / world  # per GPU
        traffic, traffic_note = None, "no ncu --set full capture of this kernel at this size is committed"
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            ent = tj.get(KERNEL_NAMES.get(kernel_used, ""), {}).get(name)
            if ent and world == 1:
                traffic, traffic_note = ent["dram_bytes_per_launch"], ent["note"]
        except Exception:
            pass
        hbm_bytes = 24.0 * sh.n * spec.T * args.steps  # 8 B read + 16 B written per state-period (whole grid)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak" if name == "c5" else "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_desc(spec, name, world, args.exchange),
            "solve_time_s": ms / args.steps * 1e-3,
            "evals_per_step": ev_total / args.steps,
            "kernel": KERNEL_NAMES.get(kernel_used, str(kernel_used)),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "phases_s_per_step": phases,
                    "what": "sdpb_create (H2D pmf/parameter tables" +
                            (", CUDA-IPC export/attach of the shards" if world > 1 else "") +
                            ") + solve + sdpb_value + D2H of the period-1 value and policy tables into page-locked host "
                            "buffers + sdpb_destroy, wall clock; one untimed warm-up cycle first"},
            "gpu_launches": int(launches_total),
            "gpu_launches_note": "backward-induction kernels (+ the per-period transposition pass of bi_lead_q2 / bi_lead_q2m) over all ranks; "
                                 "peer copies and the two 1-CTA flag kernels per period are not counted",
            "clocks": clocks,
            "device_bytes_per_gpu": dev_bytes,
            "peer_bytes_per_period": {"out": bytes_out, "in": bytes_in} if world > 1 else None,
            "roofline": {
                "bound": "fp64", "achieved": achieved, "peak": peaks["nofma_tops"], "unit": "TFLOP/s",
                "frac": achieved / peaks["nofma_tops"] if peaks["nofma_tops"] else None, "traffic": traffic,
                "traffic_note": traffic_note,
                "what": "non-fused fp64 instructions (DADD/DMUL; Java parity forbids DFMA) the kernel executes "
                        "per GPU per second vs the same mix measured live by sdpb_microbench on this GPU; "
                        "MEASURED_PEAKS.json has no fp64 figure; the per-evaluation instruction counts are audited "
                        "against ncu's DADD/DMUL counters in profiles/r02_fp64_audit.md",
                "fp64_instr_per_eval": fp_total / ev_total if ev_total else None,
                "reference_formulation_fp64_per_eval": REF_F.get(name, 20),
                "achieved_reference_formulation": ev_total * REF_F.get(name, 20) / (ms * 1e-3) / 1e12 / world,
                "reference_formulation_note": "SURVEY.md section 8(d) counts the fp64 operations of the reference's own "
                                              "lambdas per evaluation (F_A = 20, F_B = 20, F_C = 41); evals x F / t is "
                                              "above the pipe peak because the kernels remove most of those operations "
                                              "exactly -- it is NOT a utilisation; `achieved` / `frac` count only "
                                              "instructions actually issued",
                "lds_peak_gbs": peaks["lds_gbs"], "fma_peak_tflops": peaks["fma_tflops"],
                "hbm": {"achieved_gbs": hbm_bytes / (ms * 1e-3) / 1e9 / world, "peak_gbs": mp.get("hbm_gbs"),
                        "note": "algorithmic HBM bytes: 24 B per state-period; not the bound"},
            },
        }
        if kernel_used == 14:
            # bi_lead_q2m executes ~3.0 fp64 instructions per evaluation where bi_lead_q2 executed 4.125: the solve is
            # faster and `frac` -- instructions ISSUED over the pipe's rate -- is lower.  Its second limit is the SM's
            # shared-memory pipe: five 16-byte loads per thread and demand step (16 evaluations).
            lds_gbs = value * 5.0 / 1e9 / world
            out["roofline"]["shared_memory"] = {
                "achieved_gbs": lds_gbs, "peak_gbs": peaks["lds_gbs"],
                "frac": lds_gbs / peaks["lds_gbs"] if peaks["lds_gbs"] else None,
                "note": "80 B of LDS.128 per thread per demand step = 5 B per evaluation (products p*(fv+L) tabulated once "
                        "per CTA, row offsets, p*gamma) against sdpb_microbench's LDS.128 rate; ncu: fp64 pipe 68 % and "
                        "L1/shared data pipe 75 % busy at the same time (profiles/r02_c4_q2m_mix.txt)"}
            out["roofline"]["frac_note"] = (
                "round-2 kernel before the products were shared (bi_lead_q2, 4.125 fp64 instructions per evaluation): "
                "141.6 ms at frac 0.79; this kernel: fewer instructions per evaluation, shorter solve, lower frac. The same "
                "evaluations/s on the earlier formulation would need %.2f of the fp64 rate."
                % (value * 4.125 / 1e12 / world / peaks["nofma_tops"]))
        out.update(verify)
        if period_profile:
            out["period_profile"] = period_profile
    if world > 1:
        dist.barrier()
    sh.close()

    # ---- the other configurations, solved once each (plus the C5 size sweep), rank 0 prints ----
    configs = {}
    if not args.no_configs:
        peak = out["roofline"]["peak"] if rank == 0 else None
        jobs = [("c1", "c1", False, None), ("c2", "c2", False, None), ("c3", "c3", False, None),
                ("c4", "c4", False, None), ("c4_dedup", "c4", True, None)]
        for n_s in (10_000, 100_000, 1_000_000, 10_000_000, 100_000_000):
            jobs.append((f"c5_S{n_s:.0e}".replace("+0", ""), "c5", False, n_s))
        for name_key, cname, dedup, n_s in jobs:
            if cname == name and not dedup and n_s is None:
                continue  # the timed workload itself
            if n_s is not None:
                sp = S.configs.c5(n_states=n_s)
                shard = world > 1 and n_s >= 1_000_000
            else:
                sp = make_spec(S, cname, world, args.states_per_gpu)
                # never shard the folded solve: its exchange is the whole table and costs more than the 4 ms solve
                shard = cname in ("c3", "c4") and world > 1 and not dedup
            w = world if shard else 1
            if not shard and rank != 0:
                continue
            with torch.cuda.stream(stream):
                s3 = ShardedSolve(sp, rank if shard else 0, w, S.KERNEL_AUTO, dedup)
                csync = barrier if shard else torch.cuda.synchronize
                s3.step()  # warm (plain launches)
                csync()
                ev, evx, fp, kused, _ = per_step_counts(s3, csync)  # second solve: a CUDA graph when unsharded
                reps = 5 if (cname in ("c1", "c2", "c3", "c4") or (n_s or 10**9) <= 100_000) else (3 if (n_s or 10**9) <= 1_000_000 else 1)
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                csync()
                a0.record(stream)
                for _ in range(reps):
                    s3.step()
                a1.record(stream)
                csync()
                cms = a0.elapsed_time(a1) / reps
                if shard:
                    (cms, _, _, _), (_, ev, evx, fp) = reduce_max_sum([cms, ev, evx, fp])
                v0 = q0 = None
                if not shard:
                    v, q = s3.solver.value(1, INIT[cname])
                    v0, q0 = float(v[0]), float(q[0])
                tops = fp / (cms * 1e-3) / 1e12 / w
                verified = None
                if shard and not args.no_verify:
                    verified = verify_vs_unsharded(S, torch, dist, sp, s3, local, dedup)
                configs[name_key] = {"solve_ms": cms, "evals": ev, "evals_per_s": ev / (cms * 1e-3),
                                     "exchange": s3.exchange_kind, "verified_vs_unsharded": verified,
                                     "evals_executed": evx, "n_gpus": w, "kernel": KERNEL_NAMES.get(kused),
                                     "dedup": dedup, "fp64_tops_per_gpu": tops, "V1_init": v0, "Q1_init": q0,
                                     "device_bytes_per_gpu": s3.solver.grid.device_bytes,
                                     "peer_bytes_out_per_period": s3.bytes_out if shard else None}
                if shard:
                    dist.barrier()
                s3.close()
        if rank == 0:
            # The reference's drivers sweep hundreds of small instances (810 in CLSPTesting.java:57-61): sdpb_solve_batch
            # runs a list of independent handles as ONE CUDA graph (C-ABI entry point, no Python in the loop).
            nb = 64
            sp = make_spec(S, "c2", 1, args.states_per_gpu)
            batch = [S.Solver(sp, device=local) for _ in range(nb)]  # AUTO: a wide batch runs on the 2-D register tile
            for _ in range(3):  # plain solves, the capturing call, one replay
                S.solve_batch(batch)
            t0 = time.perf_counter()
            reps = 5
            for _ in range(reps):
                S.solve_batch(batch)
            dt = (time.perf_counter() - t0) / reps
            ev = batch[0].stats()["evals"] * nb
            configs["c2_batch64"] = {"solve_ms": dt * 1e3, "ms_per_instance": dt * 1e3 / nb, "evals": ev,
                                     "evals_per_s": ev / dt, "n_gpus": 1, "kernel": KERNEL_NAMES.get(batch[0].stats()["kernel_used"]),
                                     "note": "64 independent C2 instances through sdpb_solve_batch (one CUDA graph), wall clock",
                                     "dedup": False, "fp64_tops_per_gpu": batch[0].stats()["fp64_ops"] * nb / dt / 1e12}
            for b in batch:
                b.close()
            for c in configs.values():
                c["fp64_frac"] = c["fp64_tops_per_gpu"] / peak if peak else None
            # OPT-IN, reported on its own and never in evals/s: the collapsed solve of the 1-D inventory family
            # (G(y) per order-up-to level, then V(x) = opt_a cost(a) + G(x + a)); values within 1e-9 relative of the
            # exact kernels (observed ~1e-13), not bit-identical, never chosen by AUTO.
            sp = make_spec(S, "c5", 1, 10_000_000)
            with S.Solver(sp, device=local) as ex, S.Solver(sp, device=local, kernel=S.KERNEL_COLLAPSED) as co:  # (rank 0's GPU)
                ex.solve()
                co.solve()
                co.solve()
                t0 = time.perf_counter()
                reps = 5
                for _ in range(reps):
                    co.solve_async()
                co.sync()
                dt = (time.perf_counter() - t0) / reps
                Ve, Qe = ex.period_tables(1)
                Vc, Qc = co.period_tables(1)
                st = co.stats()
                out["collapsed_opt_in"] = {
                    "workload": "c5_S1e7 (10,000,000 states x 200 actions x 200 demands, T=4)", "solve_ms": dt * 1e3,
                    "exact_solve_ms": configs.get("c5_S1e7", {}).get("solve_ms"),
                    "evals_reference": st["evals"], "evals_executed": st["evals_executed"],
                    "max_rel_diff_V1_vs_exact_kernel": float(np.max(np.abs(Vc - Ve) / np.maximum(1.0, np.abs(Ve)))),
                    "policy_agreement_period1": float((Qc == Qe).mean()),
                    "note": "SDPB_KERNEL_COLLAPSED: opt-in, not bit-identical, not part of `value` or of any evals/s figure"}
    if rank == 0 and not args.no_configs:
        out["next_rows"] = next_rows(S, local)
    if rank == 0:
        out["configs"] = configs
        if not args.no_cpu_baseline:
            import oracle_lib as O
            cores = os.cpu_count() or 1
            base = make_spec(S, name, 1, args.states_per_gpu)
            rows = calibrate_rows(S, name, base, args.cpu_seconds)
            sample = cpu_sample_spec(S, name, base, rows)
            ev, dt = time_dense(sample)
            td_rate, td_ev, td_dt, td_rows, td_states = time_topdown(S, name, base)
            out["cpu_baseline"] = {
                "value": ev / dt, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"oracle_dense on a {O.grid(sample)[0]}-state sub-grid ({rows} inventory rows) of the "
                          f"{O.grid(base)[0]}-state workload (all actions, demands, T), {dt:.1f} s, {cores} threads; "
                          "a rate, not a full solve",
                "java_probe": java_probe(),
                "topdown_1thread": {"value": td_rate, "unit": UNIT,
                                    "sample": f"oracle_topdown (literal memoised recursion, 1 thread) from the initial state on "
                                              f"a cut-down instance ({td_states} states per period, first periods only): {td_rows} visited states, "
                                              f"{td_dt:.1f} s"},
                "note": "the reference is single-threaded Java (no JDK in the image, see java_probe): the C++ port is timed instead"}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse()
    sys.exit(run_reference(a) if a.impl == "reference" else run_gpu(a))
