"""Run by test_parity_gpu.py::test_lead_q2m_forced in a subprocess, with no test hook, with SDPB_Q2_SHARE=1 or with
SDPB_Q2_SPLIT = 2 or 4: the hooks are read once per process.  They force launch shapes of the lead-time-2 kernels onto
small random instances -- the shared-product kernel bi_lead_q2m without action slices (normally taken by large grids only),
or bi_lead_q2 with 2 or 4 thread groups -- and the tables are compared with the oracle over the whole grid, unsharded and
as a three-shard group (partial rows at the block ends, peer stores from the epilogue)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as O  # noqa: E402
import sdpb200 as S  # noqa: E402


def consecutive_pmf(rng, T, D):
    rows = []
    for _ in range(T):
        d0 = int(rng.integers(0, 3))
        p = rng.dirichlet(np.ones(D))
        rows.append(np.stack([np.arange(d0, d0 + D, dtype=float), p], axis=1))
    return rows


def main():
    O.load()
    rng = np.random.default_rng(20260)
    split = os.environ.get("SDPB_Q2_SPLIT")
    n = shared = 0
    for D in (1, 3, 9, 10, 11, 19, 20, 25):
        for rep in range(int(os.environ.get("SDPB_Q2M_REPS", "2"))):  # raise for a one-off campaign
            T = int(rng.integers(2, 4))
            spec = S.leadtime_model(consecutive_pmf(rng, T, D), fixed_cost=float(rng.integers(0, 9)),
                                    vari_cost=float(rng.integers(0, 3)) + 0.25 * rep, hold_cost=float(rng.integers(1, 4)),
                                    penalty_cost=float(rng.integers(2, 12)),
                                    max_order=int(rng.integers(30, 61)) if rep % 2 == 0 else int(rng.integers(1, 30)),
                                    inv_min=-float(rng.integers(2, 12)), inv_max=float(rng.integers(3, 14)), lead_time=2,
                                    clamp=True)
            Vo, Qo, evals, _ = O.dense(spec)
            with S.Solver(spec, kernel=S.KERNEL_LEAD_Q2) as s:
                s.solve()
                used = s.stats()["kernel_used"]   # tiny order ranges (tables larger than the budget) stay on bi_lead_q2
                assert used == S.KERNEL_LEAD_Q2 if split else used in (S.KERNEL_LEAD_Q2, S.KERNEL_LEAD_Q2M), (used, split)
                shared += used == S.KERNEL_LEAD_Q2M
                for t in range(1, spec.T + 1):
                    V, Q = s.period_tables(t)
                    assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), (D, rep, t, spec)
                assert s.stats()["evals"] == evals
            with S.Group(spec, [0, 0, 0], kernel=S.KERNEL_LEAD_Q2) as g:
                g.solve()
                for t in range(1, spec.T + 1):
                    V, Q = g.period_tables(t)
                    assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), ("group", D, rep, t, spec)
            n += 1
    if not split:
        assert shared >= 8, shared   # (the wide order ranges of rep 0 always fit the shared-memory budget)
    print(f"q2m worker: {n} instances ok, {shared} on the shared-product kernel (SDPB_Q2_SHARE={os.environ.get('SDPB_Q2_SHARE', '-')}, "
          f"SDPB_Q2_SPLIT={split or '-'})")


if __name__ == "__main__":
    main()
