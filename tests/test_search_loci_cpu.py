"""The loci of search_loci.py do what the GPU search tests (test_gpu_search_range.py) need them to do, checked with the CPU
oracle: every search climbs to a state of max_causal SNPs (so that searches with c >= 6 score 6-8 SNP neighbourhoods on
score_batch_kernel), the round-100 cases stop by the reference's convergence rule with new configurations in that round
and a criterion far from its threshold, and the prior arithmetic behind the lane kernel's admission test."""
import math

import numpy as np
import pytest

import search_loci as S
from conftest import synth_as_oracle_locus


def _oracle_search(name, max_iter=1000):
    from oracle import oracle as O
    SL, c = S.search_locus(name)
    return SL, c, O.sss(synth_as_oracle_locus(SL), c, max_iter=max_iter)


@pytest.mark.parametrize("name", sorted(S.SEARCHES))
def test_search_reaches_max_causal(name):
    SL, c, want = _oracle_search(name)
    _, _, _, rounds, why = S.SEARCHES[name]
    assert (want.extra["n_iter"], S.stop_reason(want)) == (rounds, why)
    sizes = [len(s) for s in S.states(SL.U, c, want.extra["trace"])]
    assert max(sizes) == c
    if c >= 6:                                  # several rounds score neighbourhoods of c-SNP configurations
        assert sum(k >= c - 1 for k in sizes) >= 5


@pytest.mark.parametrize("name", [n for n in sorted(S.SEARCHES) if S.SEARCHES[n][4] == 2])
def test_round_100_ends_by_convergence(name):
    """The reference consults its running total from round 100 on (sss_postcal.cpp:265-270): these searches stop there by
    that rule, not because a round found nothing new, and 1 - exp(total_99 - total_100) sits far below 0.001, so that the
    order in which the GPU adds its terms cannot move the stop."""
    from oracle import oracle as O
    SL, c, want = _oracle_search(name)
    tr = want.extra["trace"]
    assert want.extra["n_iter"] == 100 and tr[100, 2] > 0
    L = synth_as_oracle_locus(SL)
    t99, t100 = O.sss(L, c, max_iter=100).total, O.sss(L, c, max_iter=101).total
    assert t100 == want.total
    crit = 1.0 - math.exp(t99 - t100)
    assert 0.0 <= crit < 0.0005, crit


def test_capped_search_is_a_prefix():
    """max_iterations inside a round-100 search: stop reason 0 and the accumulators of the first 60 rounds."""
    SL, c, want = _oracle_search("c7_round100", max_iter=60)
    assert want.extra["n_iter"] == 60 and S.stop_reason(want, 60) == 0


def test_every_neighbour_scores_minus_inf_at_p1():
    """At p = 1 every expansion that puts a SNP in one study only has prior 0, and every non-empty configuration has such an
    expansion: its largest-|l| value is -inf, and the search would weigh its groups by nan.  The engine refuses a search
    there (test_gpu_search_range.py)."""
    from oracle import oracle as O
    SL, _ = S.search_locus("c5")
    L = synth_as_oracle_locus(S.with_prior(SL, p=1.0))
    idx = np.full((1 + SL.U, 2), -1, dtype=np.int32)
    idx[1:, 0] = np.arange(SL.U)
    idx[2:, 1] = np.arange(1, SL.U)[::-1]
    idx[2:] = np.sort(idx[2:], 1)
    idx[2:][idx[2:, 0] == idx[2:, 1], 1] = -1
    m, _ = O.score_union_configs(L, idx)
    assert np.isfinite(m[0]) and np.all(np.isneginf(m[1:]))


def test_lane_admission_rho_alone():
    """The old admission test looked at rho^8 only: a normal double with a finite reciprocal.  The cutoff is p ~ 1.5e-39."""
    assert S.lane_ok_rho_only(1e-38) and S.lane_ok_rho_only(2e-39)
    assert not S.lane_ok_rho_only(1e-40)
    assert S.lane_ok_rho_only(0.0) and S.lane_ok_rho_only(0.999999) and not S.lane_ok_rho_only(1.0)


def test_lane_weight_overflows_where_rho_alone_admits():
    """w0[1] = pi'(5, 0) / rho^4 times a table entry just inside the fast range (2^449.99), computed as lane_score<5>
    computes it: inf at gamma = 0.99999 and p = 2e-39 although rho^8 is a normal double; finite at 0.9999 and 0.5."""
    E = 2.0 ** 449.99
    with np.errstate(over="ignore"):
        big = S.lane_weights(0.99999, 2e-39, 5, 5)[0][1] * np.float64(E)
        mid = S.lane_weights(0.9999, 2e-39, 5, 5)[0][1] * np.float64(E)
        low = S.lane_weights(0.5, 2e-39, 5, 5)[0][1] * np.float64(E)
    assert S.lane_ok_rho_only(2e-39)
    assert np.isinf(big)
    assert 1e307 < mid < 1e308 and 1e287 < low < 1e288
    # the admission test now bounds every value the kernel forms: such priors go to score_batch_kernel
    assert not S.lane_ok(0.99999, 2e-39) and not S.lane_ok(0.9999, 2e-39)
    assert S.lane_ok(0.5, 2e-39) and S.lane_ok(0.01, 1e-38) and not S.lane_ok(0.01, 1e-40)
    for g in (1e-6, 0.01, 0.5):
        for p in (0.0, 1e-9, 0.2, 1 / 3, 0.75, 0.999999):
            assert S.lane_ok(g, p), (g, p)
