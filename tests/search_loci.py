"""Loci on which the stochastic shotgun search (pipsort_sss, sss_postcal.cpp:102-380) climbs to states of max_causal SNPs,
and the scoring kernels' routing by the prior restated in float64.

The search draws inside each neighbourhood group (zero / minus / plus) relative to the group's own best value, and then
across the groups by their summed weights.  On a locus with one or two strong SNPs every group is dominated by one
configuration, the weights of the groups are ~1 each, and the walk falls back to the empty state within a few rounds.
With nearly flat likelihoods every neighbour counts: the group weights act like the group sizes, the plus group (U - k
neighbours) outweighs the minus group (k), and the walk climbs until it holds max_causal SNPs.  Such loci reach the
6-8 SNP states that the lane kernel (score_lane.cuh, <= 5 SNPs per configuration) hands to score_batch_kernel, and some
of them run long enough for the reference's convergence rule of round 100.

Test infrastructure only (numpy + the CPU oracle).
"""
from __future__ import annotations

import dataclasses

import numpy as np

from pipsort_b200 import synth

LANE_KMAX = 5           # score_lane.cuh: the most SNPs per configuration of the lane kernel
FAST_BITS = 450.0       # every table entry E_s(mask) of the lane kernel's plain-double path is < 2^450


def flat_locus(n, overlap, seed, scale):
    """synth.make_locus(n, overlap, seed) with each study's z replaced by scale * chol(LD) @ N(0, I) (no causal SNP; the
    z-scores fit the LD) and K = sum_s z' LD^-1 z recomputed.  Sample sizes of 1000 in both studies keep d small."""
    SL = synth.make_locus(n, overlap=overlap, seed=seed, sample_sizes=(1000, 1000))
    rng = np.random.default_rng(seed)
    z, K = [], 0.0
    for s in range(2):
        C = np.linalg.cholesky(np.asarray(SL.sigma[s]))
        v = scale * (C @ rng.standard_normal(int(SL.num_snps[s])))
        y = np.linalg.solve(C, v)
        z.append(v)
        K += float(y @ y)
    return dataclasses.replace(SL, z=z, K=K)


def with_prior(SL, gamma=None, p=None):
    """The same locus under another prior (gamma, sharing parameter p)."""
    return dataclasses.replace(SL, gamma=SL.gamma if gamma is None else gamma,
                               sharing_param=SL.sharing_param if p is None else p)


# ---- what the oracle's search did -------------------------------------------------------------------------------------
def neighbourhood(cur, U, c):
    """zero ++ minus ++ plus of a sorted union configuration (sss_postcal.cpp:20-99,166-186)."""
    cur = list(cur)
    non = [g for g in range(U) if g not in set(cur)]
    minus = [cur[:m] + cur[m + 1:] for m in range(len(cur))]
    zero = [sorted(m + [g]) for g in non for m in minus]
    plus = [sorted(cur + [g]) for g in non] if len(cur) < c else []
    return zero + minus + plus


def states(U, c, trace):
    """The current state of every round of an oracle search, replayed from its trace (column 1 = neighbourhood size,
    column 3 = index of the neighbour drawn)."""
    cur, out = [], []
    for row in trace:
        out.append(cur)
        nbd = neighbourhood(cur, U, c)
        assert len(nbd) == row[1]
        if row[3] >= 0:
            cur = nbd[row[3]]
    return out


def stop_reason(want, max_iter=1000):
    """pipsort_sss's stop reason of an oracle search: 0 = iteration cap, 1 = a round without new configurations
    ("hit break condition"), 2 = convergence (the round-100 rule)."""
    it, trace = want.extra["n_iter"], want.extra["trace"]
    if it == max_iter:
        return 0
    return 1 if trace[it, 2] == 0 else 2


# ---- the prior weights of the lane kernel -----------------------------------------------------------------------------
def rho(p):
    """pi'(k, a) = pi'(k, 0) rho^a (engine.cu)."""
    return 1.0 if p == 0.0 else p / ((1.0 - p) * 0.5)


def pi0(gamma, p, k):
    """pi'(k, 0) = (gamma / (1 - gamma))^k ((1 - p) / 2)^k; the sharing term is left out at p = 0 (postcal.cpp:27)."""
    r = (gamma / (1.0 - gamma)) ** k
    return r if p == 0.0 else r * ((1.0 - p) * 0.5) ** k


def lane_ok_rho_only(p):
    """The lane kernel's original admission test (engine.cu): rho^8 finite, non-zero, with a finite reciprocal."""
    if not p < 1.0:
        return False
    with np.errstate(over="ignore", under="ignore"):
        r8 = np.float64(rho(p)) ** 8
        return bool(np.isfinite(r8) and r8 > 0.0 and np.isfinite(1.0 / r8))


def lane_weights(gamma, p, k, K):
    """w0[j] = pi'(k, 0) rho^(j - K) and w1[j] = rho^j, j = 0..K, as lane_score<K> forms them for a row of k SNPs."""
    with np.errstate(over="ignore", under="ignore"):
        w1 = [np.float64(1.0)]
        for _ in range(K):
            w1.append(w1[-1] * np.float64(rho(p)))
        cx = np.float64(pi0(gamma, p, k)) / w1[K]
        return [cx * w for w in w1], w1


def lane_peak_bits(gamma, p):
    """engine.cu lane_peak_bits restated: log2 of the largest value lane_score forms under the prior, over rows of k SNPs
    in warp-steps of K >= k SNPs (K <= LANE_KMAX): the weights w0[j], w1[j] times a table entry (1 for the empty mask,
    up to 2^450 otherwise), the terms pi'(k, 0) rho^a E_0 E_1 (0 <= a <= k), plus 2 LANE_KMAX bits for the sums."""
    lr = float(np.log2(rho(p)))
    peak = -np.inf
    for K in range(1, LANE_KMAX + 1):
        for k in range(1, K + 1):
            lp = float(np.log2(pi0(gamma, p, k)))
            for j in range(K + 1):
                e = FAST_BITS if j > 0 else 0.0
                peak = max(peak, max(lp + (j - K) * lr, j * lr) + e)
            for a in range(k + 1):
                peak = max(peak, lp + a * lr + 2 * FAST_BITS)
    return peak + 2 * LANE_KMAX


def lane_ok(gamma, p):
    """The lane kernel's admission test (engine.cu): rho^8 a normal double and every value it forms below 2^1000."""
    return lane_ok_rho_only(p) and lane_peak_bits(gamma, p) < 1000.0


# ---- the searches the GPU tests run ---------------------------------------------------------------------------------
# name: (flat_locus arguments (n, overlap, seed, scale), sharing parameter, max_causal, rounds, stop reason) as the CPU
# oracle runs them; test_search_loci_cpu.py checks these outcomes and that every search reaches a state of max_causal SNPs.
SEARCHES = {
    "c0": ((16, 0.6, 3, 0.3), 0.75, 0, 0, 1),
    "c1": ((16, 0.6, 3, 0.3), 0.75, 1, 2, 1),
    "c2": ((16, 0.6, 3, 0.3), 0.75, 2, 8, 1),
    "c5": ((16, 0.6, 3, 0.3), 0.75, 5, 67, 1),
    "c6": ((16, 0.6, 3, 0.3), 0.75, 6, 36, 1),
    "c7_round100": ((16, 0.6, 3, 0.3), 0.75, 7, 100, 2),
    "c8_round100": ((16, 0.6, 3, 0.3), 0.75, 8, 100, 2),
    "c8_seed4": ((16, 0.6, 4, 0.3), 0.75, 8, 100, 2),
    "c6_round100": ((16, 0.6, 7, 0.3), 0.75, 6, 100, 2),
    "p0_c4": ((16, 0.6, 4, 0.3), 0.0, 4, 73, 1),
}


def search_locus(name):
    args, p, c, _, _ = SEARCHES[name]
    return with_prior(flat_locus(*args), p=p), c
