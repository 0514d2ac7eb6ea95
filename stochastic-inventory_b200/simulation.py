"""Host-side mirror of the reference's policy roll-out classes, over sdpb_simulate (a dense recursion),
sdpb_topdown_simulate (a recursion built with topdown=True) or sdpb_reached_simulate (a reached-state engine:
CashRecursionMultiLead, CashRecursionMultiXR, CashRecursionV, CashRecursionRounded).

    Simulation       src/sdp/inventory/Simulation.java:19-107
    CashSimulation   src/sdp/cash/CashSimulation.java:30-118

The reference draws its Latin-hypercube samples with Math.random() (src/sdp/sampling/Sampling.java:94),
so its simulated means are not reproducible run to run; here the sample matrix is an explicit argument
(from sampling.Sampling, the MRG32k3a mirror of Sampling.java, or from `generate_lh_samples`, a vectorised
numpy generator with the same stratified scheme), and the roll-out itself —
Q = getAction(state); d = Math.round(sample); sum += c; state = f — runs on the GPU, one thread per path.
"""
from __future__ import annotations

import numpy as np


def generate_lh_samples(distributions, sample_num, seed=20261018):
    """Sampling.generateLHSamples (Sampling.java:86-103): one stratum per sample and period, a uniform
    draw inside it, inverse cdf, then a shuffle of each column."""
    rng = np.random.default_rng(seed)
    T = len(distributions)
    out = np.empty((sample_num, T))
    for i, dist in enumerate(distributions):
        u = (np.arange(sample_num) + rng.random(sample_num)) / sample_num
        col = np.array([dist.inverseF(x) for x in u])
        rng.shuffle(col)
        out[:, i] = col
    return out


class Simulation:
    """new Simulation(distributions, sampleNum, recursion) — Simulation.java:34-41."""
    discountFactor = 1.0

    def __init__(self, distributions, sampleNum, recursion, discountFactor=1.0):
        self.distributions = list(distributions)
        self.sampleNum = int(sampleNum)
        self.recursion = recursion
        self.discountFactor = float(discountFactor)

    def setSampleNum(self, n):
        self.sampleNum = int(n)

    def simulate_paths(self, iniState, samples=None):
        """Per-path sums (the reference's simuValues array)."""
        if samples is None:
            samples = generate_lh_samples(self.distributions, self.sampleNum)
        self.recursion.getExpectedValue(iniState)  # solves on first use, like the reference's lazy recursion
        if getattr(self.recursion, "_rh", None) is not None:
            # a two-product (reached-state) engine: samples are [n, T, 2] (one demand per product), or [n, T] for one
            return self.recursion._rh.simulate(iniState._vec(), samples, self.discountFactor)
        if getattr(self.recursion, "_topdown", False):
            # no grid: the roll-out solves each state a path meets that was not reached yet (Simulation.java:62)
            return self.recursion._td.simulate(iniState._vec(), samples, self.discountFactor)
        return self.recursion._solver.simulate(iniState._vec(), samples, self.discountFactor)

    def simulateSDPGivenSamplNum(self, iniState, samples=None):
        vals = self.simulate_paths(iniState, samples)
        return float(vals.sum() / len(vals))


class CashSimulation(Simulation):
    """CashSimulation.java:49-57,85-118: discounted sums, mean + iniCash."""

    def simulateSDPGivenSamplNum(self, iniState, samples=None):
        vals = self.simulate_paths(iniState, samples)
        return float(vals.sum() / len(vals)) + iniState.getIniCash()
