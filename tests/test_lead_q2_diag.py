"""bi_lead_q2m walks each action's demand loop along level diagonals, with three preQ2 columns per thread.  These
instances cover what that shape depends on: nQ in every residue class mod 3 (the column stride) and mod 8 (the chunk of
preQ1 slots), demand supports of 1 to 17 points (shorter than, equal to and longer than the 7 diagonals at each end, and
every remainder of the 8-step main loop), MIN and MAX, backorders and lost sales, one handle and a three-shard group
whose blocks end inside inventory rows.  Every period's tables must equal the oracle's.

The launch shape is chosen once per process (SDPB_Q2_SHARE), so each mode runs this file as a script in a subprocess:
by default these small grids cut the action range over separate CTAs and merge the slices; SDPB_Q2_SHARE=1 runs one
CTA per block of states over all actions and stores the peers' rows from the kernel's epilogue."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def consecutive_pmf(rng, T, D):
    rows = []
    for _ in range(T):
        d0 = int(rng.integers(0, 3))
        p = rng.dirichlet(np.ones(D))
        rows.append(np.stack([np.arange(d0, d0 + D, dtype=float), p], axis=1))
    return rows


def main():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    import sdpb200 as S
    A = S.abi
    O.load()
    rng = np.random.default_rng(31)
    n = 0
    for D in range(1, 18):
        nQ = 34 + D % 8                        # 34..41: every class mod 8, and mod 3
        T = int(rng.integers(2, 4))
        spec = S.leadtime_model(consecutive_pmf(rng, T, D), fixed_cost=float(rng.integers(0, 9)),
                                vari_cost=float(rng.integers(0, 3)) + 0.5, hold_cost=float(rng.integers(1, 4)),
                                penalty_cost=float(rng.integers(2, 12)), max_order=nQ - 1,
                                inv_min=-float(rng.integers(4, 10)), inv_max=float(rng.integers(4, 10)), lead_time=2,
                                clamp=True)
        if D % 2:
            spec.direction = A.MAX
        if (D // 2) % 2:
            spec.flags |= A.F_LOST_SALES
        Vo, Qo, evals, _ = O.dense(spec)
        with S.Solver(spec, kernel=S.KERNEL_LEAD_Q2) as s:
            s.solve()
            st = s.stats()
            assert st["kernel_used"] == S.KERNEL_LEAD_Q2M, (D, nQ, st["kernel_used"])
            assert st["evals"] == evals
            for t in range(1, spec.T + 1):
                V, Q = s.period_tables(t)
                assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), (D, nQ, t)
        with S.Group(spec, [0, 0, 0], kernel=S.KERNEL_LEAD_Q2) as g:
            g.solve()
            for t in range(1, spec.T + 1):
                V, Q = g.period_tables(t)
                assert np.array_equal(V, Vo[t - 1]) and np.array_equal(Q, Qo[t - 1]), ("group", D, nQ, t)
        n += 1
    print(f"diagonal q2m: {n} instances ok (SDPB_Q2_SHARE={os.environ.get('SDPB_Q2_SHARE', '-')})")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["sliced", "share"])
def test_lead_q2m_diagonals(mode):
    env = dict(os.environ)
    env.pop("SDPB_Q2_SHARE", None), env.pop("SDPB_Q2_SPLIT", None)
    if mode == "share":
        env["SDPB_Q2_SHARE"] = "1"
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "17 instances ok" in r.stdout


if __name__ == "__main__":
    main()
