"""Stochastic shotgun search with the device-resident search state (pipsort_sss; sss_postcal.cpp:102-380) against
17-digit dumps of the reference's own `-q 1` runs, the oracle's restatement of the search, and -- at the size of
BASELINE.json configs[4] (5000 SNPs per study, c = 5) -- sampled neighbours against the oracle plus size-independent
properties of one batched neighbourhood."""
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import (GOLDEN, args_to_params, assert_results_match, engine_for, golden, oracle_locus, synth_as_oracle_locus,
                      synth_locus)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["small_sss_c3_p075", "small_sss_c2_p025", "example_sss_c2_p025"])
def test_sss_matches_reference_dump(name):
    from oracle import oracle as O
    g = golden(name)
    prm = args_to_params(g["args"])
    L = oracle_locus(g["dataset"], p=prm["p"], gamma=prm["gamma"], s=prm["s"], t=prm["t"])
    with engine_for(L, prm["c"]) as e:
        r, iters, why = e.sss(prm["c"])
    assert_results_match(r, g)
    want = O.sss(L, prm["c"])
    assert iters == want.extra["n_iter"]                 # same trajectory: same number of rounds
    assert (why == 1) == any("hit break condition" in f for f in g["stdout_flags"])
    assert (why == 2) == any("hit convergence condition" in f for f in g["stdout_flags"])


def test_sss_synthetic_matches_oracle_trajectory():
    """60+60 SNPs with mixed SNP types, c = 4: several hundred rounds of the search, every draw identical to the oracle's
    (std::mt19937(12345) + std::discrete_distribution on the same doubles), so the accumulators agree to 1e-10."""
    from oracle import oracle as O
    from pipsort_b200 import synth
    L = synth.make_locus(60, overlap=0.7, seed=21)
    want = O.sss(synth_as_oracle_locus(L), 4, max_iter=60)
    with engine_for(L, 4) as e:
        r, iters, why = e.sss(4, max_iterations=60)
    assert iters == want.extra["n_iter"]
    assert_results_match(r, want)


def test_sss_convergence_rule_reads_the_running_total():
    """The convergence rule (sss_postcal.cpp:265-270) compares the running totals after consecutive rounds.  The reference
    starts it at round 100, which a search on this locus never reaches (test_gpu_search_range.py runs searches that stop
    there); PIPSORT_SSS_CONV_FROM=2 starts it at round 2.  On 12+12 SNPs
    (c = 3, 9 rounds to the break condition) the totals the engine reports after k = 1..9 rounds predict the round at which
    the rule stops the search."""
    from pipsort_b200 import synth
    SL = synth.make_locus(12, overlap=0.7, seed=18)
    with engine_for(SL, 3) as e:
        total = [None]                                   # total[k]: after k rounds
        for k in range(1, 10):
            r, iters, why = e.sss(3, max_iterations=k)
            assert (iters, why) == (k, 0)
            total.append(r.total)
        # round i (counted from 0) stops the search when i >= 2 + 1 and 1 - exp(total[i] - total[i + 1]) <= 0.001
        crit = {i: 1 - math.exp(total[i] - total[i + 1]) for i in range(3, 9)}
        stops = [i for i in crit if crit[i] <= 0.001]
        assert stops
        stop = stops[0]
        for i in range(3, stop + 1):                     # accumulation order varies: no round may sit on the threshold
            assert abs(crit[i] - 0.001) > 1e-6, (i, crit[i])
        os.environ["PIPSORT_SSS_CONV_FROM"] = "2"
        try:
            _, iters, why = e.sss(3)
        finally:
            os.environ.pop("PIPSORT_SSS_CONV_FROM", None)
    assert (iters, why) == (stop, 2)


def test_host_loop_and_device_state_agree_through_the_cli():
    """PIPSORT_SSS_HOSTLOOP=1 keeps the neighbourhood lists and the std::map on the host (independently written);
    both must write the reference's six files byte for byte."""
    from pipsort_b200 import build
    build.build_engine()
    exe = build.build_host()
    g = golden("example_sss_c2_p025")
    d = os.path.join(GOLDEN, "example")
    for env_extra in ({}, {"PIPSORT_SSS_HOSTLOOP": "1"}):
        with tempfile.TemporaryDirectory() as tmp:
            out = os.path.join(tmp, "o")
            p = subprocess.run([exe, "-l", "ldfiles.txt", "-z", "zfiles.txt", "-m", "snp_map", "-n", g["sample_sizes"], "-o", out]
                               + g["args"], cwd=d, capture_output=True, text=True, env=dict(os.environ, **env_extra))
            assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
            for suf, want in g["files"].items():
                with open(f"{out}_{suf}.txt") as f:
                    assert f.read() == want, (env_extra, suf)


def neighbourhood(cur, U, c):
    """zero ++ minus ++ plus of a sorted union configuration (sss_postcal.cpp:20-99,166-186)."""
    cur = list(cur)
    non = [g for g in range(U) if g not in set(cur)]
    minus = [cur[:m] + cur[m + 1:] for m in range(len(cur))]
    zero = [sorted(m + [g]) for g in non for m in minus]
    plus = [sorted(cur + [g]) for g in non] if len(cur) < c else []
    return zero + minus + plus


def test_config_d_neighbourhood_5000_snps_c5():
    """BASELINE.json configs[4]: 5000 SNPs/study (U = 6000), c = 5.  One neighbourhood of a 4-SNP state = 29,984 union
    configurations x up to 3^5 expansions in ONE launch; 48 sampled neighbours are checked against the oracle, the
    whole batch through additivity (two half batches == the full batch) and idempotence of re-reading."""
    from oracle import oracle as O
    from pipsort_b200 import synth
    L = synth_locus(5000)
    U, c = L.U, 5
    assert U == 6000
    strong = [int(np.argmax(np.abs(L.z[0])))]
    cur = sorted({int(np.where(L.snp_map[0] == strong[0])[0][0]), 17, 2999, 5998})
    nbd = neighbourhood(cur, U, c)
    assert len(nbd) == (U - 4) * 4 + 4 + (U - 4) == 29984
    idx = np.full((len(nbd), c), -1, dtype=np.int32)
    for i, v in enumerate(nbd):
        idx[i, :len(v)] = v
    with engine_for(L, c) as e:
        got = e.score_union_configs(idx)
        full = e.read()
        e.reset()
        a = e.score_union_configs(idx[:15000])
        b = e.score_union_configs(idx[15000:])
        halves = e.read()
    np.testing.assert_array_equal(np.concatenate([a, b]), got)
    assert_results_match(halves, full, rtol=1e-12)
    assert full.n_configs == sum(3 ** int(((L.snp_map[0][v] >= 0) & (L.snp_map[1][v] >= 0)).sum()) for v in map(np.array, nbd))
    rng = np.random.default_rng(1)
    pick = np.sort(rng.choice(len(nbd), 48, replace=False))
    want_l, _ = O.score_union_configs(synth_as_oracle_locus(L), idx[pick])
    np.testing.assert_allclose(got[pick], want_l, rtol=1e-10)


def test_config_d_sample_batch_accumulators_against_oracle():
    """BASELINE.json configs[4] again: 384 neighbours sampled from the same 29,984-configuration neighbourhood (plus the
    null configuration and the current state), scored as ONE batch on fresh accumulators -- every accumulator (total,
    postValues, noCausal, sharedPips, sharedLL, notSharedLL) and every max-|l| value against the oracle's
    expand_and_compute_lkl restatement (sss_postcal.cpp:447-685), with make_updates off for a quarter of the rows."""
    from oracle import oracle as O
    L = synth_locus(5000)
    U, c = L.U, 5
    strong = int(np.where(L.snp_map[0] == int(np.argmax(np.abs(L.z[0]))))[0][0])
    cur = sorted({strong, 17, 2999, 5998})
    nbd = neighbourhood(cur, U, c)
    rng = np.random.default_rng(5)
    pick = np.sort(rng.choice(len(nbd), 384, replace=False))
    rows = [[], cur] + [nbd[i] for i in pick]
    idx = np.full((len(rows), c), -1, dtype=np.int32)
    for i, v in enumerate(rows):
        idx[i, :len(v)] = v
    upd = (rng.uniform(size=len(rows)) < 0.75).astype(np.uint8)
    upd[:2] = 1
    want_l, want = O.score_union_configs(synth_as_oracle_locus(L), idx, upd)
    with engine_for(L, c) as e:
        got_l = e.score_union_configs(idx, upd)
        got = e.read()
    np.testing.assert_allclose(got_l, want_l, rtol=1e-10, atol=0)
    assert_results_match(got, want)


def test_bad_union_configuration_is_refused():
    """pipsort_score_union_configs validates its rows like the explicit-configuration path does: an index >= U, a repeated
    or a descending index raise PIPSORT_E_CONFIG instead of reading out of bounds / scoring a different configuration."""
    import pipsort_b200 as P
    L = oracle_locus("small_example")
    for row in ([3, 3, -1], [5, 2, -1], [1, L.U, -1], [0, 1, 40000]):
        with engine_for(L, 3) as e:
            with pytest.raises(P.PipsortError) as ei:
                e.score_union_configs(np.array([[0, 4, 7], row], dtype=np.int32))
                e.read()
            assert ei.value.code == 6
