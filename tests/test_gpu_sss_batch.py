"""The shotgun search for a list of loci in one call (pipsort_sss_batch), against one-at-a-time pipsort_sss on the same loci,
the golden dumps of the reference's own -q 1 runs and the oracle's search.

* The golden dumps inside batches of other loci.
* 40 distinct loci -- the flat loci of search_loci.py, which climb to states of max_causal SNPs, and synthetic loci with
  mixed SNP types, three gammas and sharing parameters from 0 up -- at c = 0, 1, 2, 5, 6, 7 and 8: rounds and stop reason
  equal exactly, every output to 1e-12 relative (the kernels and the draws are the same; only the order of the atomics
  differs), and each flat locus at its own c equal to the oracle's search, trajectory and accumulators.
* The same argument block three times, and at other depths; 1, 2 and 8 host threads in child processes
  (PIPSORT_BATCH_THREADS is read once per process).
* One bad locus at position 17 of 40, refused before the search or found during it: the error reaches the caller, a
  refusal names the locus, the memory pool is back at its baseline and the next batch is right.

Before every run() the outputs are filled with NaN and the per-locus counts with sentinels.
"""
import copy
import dataclasses
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

import search_loci as S
from conftest import ROOT, args_to_params, assert_results_match, engine_for, golden, oracle_locus
from test_gpu_batch import GAMMAS, OVERLAPS, SHARING, as_dict, as_oracle, assert_each, expect_error, pool_used  # noqa: F401
from test_gpu_search_range import oracle_search

pytestmark = pytest.mark.gpu

PIPSORT_E_ARG, PIPSORT_E_RANGE, PIPSORT_E_SINGULAR = 1, 4, 5
RTOL_SAME = 1e-12
CS = (0, 1, 2, 5, 6, 7, 8)
# the distinct loci of search_loci.SEARCHES (several searches there share a locus): 4, at p = 0.75 and p = 0
FLAT = sorted({S.SEARCHES[n][:2] for n in S.SEARCHES})


@functools.lru_cache(maxsize=None)
def loci():
    """40 distinct loci: the flat loci of search_loci.py, then 36 synthetic loci of 12 .. 40 SNPs per study with the
    overlaps, gammas and sharing parameters of test_gpu_batch in turn (p = 0 among them)."""
    from pipsort_b200 import synth
    out = [S.with_prior(S.flat_locus(*args), p=p) for args, p in FLAT]
    out += [synth.make_locus(12 + 28 * i // 35, overlap=OVERLAPS[i % 4], seed=700 + i, gamma=GAMMAS[i % 3],
                             sharing_param=SHARING[i % 5]) for i in range(40 - len(FLAT))]
    return out


def run_fresh(B):
    """B.run() into outputs of NaN and sentinel counts; (Results per locus, iterations, stop reasons), copied out."""
    B.buf.fill(np.nan)
    B.cnt[:] = 0
    B.iterations[:] = -1
    B.stop_reasons[:] = -1
    B.run()
    return copy.deepcopy(B.results()), B.iterations.copy(), B.stop_reasons.copy()


def batch(D, c, **kw):
    import pipsort_b200 as P
    return run_fresh(P.LocusBatch(D, c, search=True, **kw))


@functools.lru_cache(maxsize=None)
def one_at_a_time(c):
    """pipsort_sss on a fresh engine per locus (max_causal = c at create, as LocusBatch creates them)."""
    out = []
    for L in loci():
        with engine_for(L, c) as e:
            out.append(e.sss(c))
    return out


def same_search(got, want):
    """got: (Results, iterations, stop reason) of the batch, want: of Engine.sss."""
    r, it, why = got
    wr, wit, wwhy = want
    assert (it, why) == (wit, wwhy)
    assert r.n_configs == wr.n_configs
    assert_results_match(r, wr, rtol=RTOL_SAME)


def check_against_one_at_a_time(out, c):
    res, it, why = out
    assert_each(list(zip(res, it.tolist(), why.tolist())), one_at_a_time(c), same_search)


# ---- 1. the reference's own searches -------------------------------------------------------------------------------------
def golden_case(name):
    g = golden(name)
    prm = args_to_params(g["args"])
    return g, prm, oracle_locus(g["dataset"], p=prm["p"], gamma=prm["gamma"], s=prm["s"], t=prm["t"])


@pytest.mark.parametrize("c,names", [(2, ("small_sss_c2_p025", "example_sss_c2_p025")), (3, ("small_sss_c3_p075",))])
def test_reference_dumps_inside_a_batch(c, names):
    """Each dump between synthetic loci in a batch of 10 (three threads): results equal the dump, the stop reason the one
    the reference printed, the rounds those of one-at-a-time pipsort_sss."""
    pad = [as_dict(L) for L in loci()[4:12]]
    cases = [golden_case(n) for n in names]
    assert all(prm["c"] == c for _, prm, _ in cases)
    D = pad[:3] + [as_dict(L) for _, _, L in cases] + pad[3:]
    res, it, why = batch(D, c)
    for k, (g, _, L) in enumerate(cases):
        r = res[3 + k]
        assert_results_match(r, g)
        assert (why[3 + k] == 1) == any("hit break condition" in f for f in g["stdout_flags"])
        assert (why[3 + k] == 2) == any("hit convergence condition" in f for f in g["stdout_flags"])
        with engine_for(L, c) as e:
            _, wit, wwhy = e.sss(c)
        assert (it[3 + k], why[3 + k]) == (wit, wwhy)


# ---- 2. 40 distinct loci ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", CS)
def test_forty_loci_match_one_at_a_time_and_the_oracle(c):
    res, it, why = out = batch([as_dict(L) for L in loci()], c)
    check_against_one_at_a_time(out, c)
    for name, (args, p, c_name, _, _) in sorted(S.SEARCHES.items()):
        if c_name != c:
            continue
        k = FLAT.index((args, p))
        want = oracle_search(name)
        assert (it[k], why[k]) == (want.extra["n_iter"], S.stop_reason(want)) == tuple(S.SEARCHES[name][3:]), name
        assert_results_match(res[k], want)


def test_same_argument_block_three_times_and_other_depths():
    """One LocusBatch called three times, then at 1 and 5 searches in flight per thread (PIPSORT_SSS_DEPTH is read at every
    call): always what one-at-a-time pipsort_sss gives."""
    import pipsort_b200 as P
    B = P.LocusBatch([as_dict(L) for L in loci()], 5, search=True)
    for _ in range(3):
        check_against_one_at_a_time(run_fresh(B), 5)
    for depth in ("1", "5"):
        os.environ["PIPSORT_SSS_DEPTH"] = depth
        try:
            out = run_fresh(B)
        finally:
            os.environ.pop("PIPSORT_SSS_DEPTH", None)
        check_against_one_at_a_time(out, 5)


def test_iteration_cap():
    """max_iterations caps every search of the list as it caps pipsort_sss; 0 runs no round and reads empty stores."""
    D = [as_dict(L) for L in loci()]
    for cap in (0, 7):
        res, it, why = batch(D, 6, max_iterations=cap)
        for k, L in enumerate(loci()):
            with engine_for(L, 6) as e:
                same_search((res[k], int(it[k]), int(why[k])), e.sss(6, max_iterations=cap))


CHILD = """
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import pipsort_b200 as P
src = np.load(sys.argv[2])
keys = ("num_snps", "sigma", "z", "d", "K", "snp_map", "gamma", "sharing_param")
loci = [{k: src[f"{k}{i}"] for k in keys} for i in range(int(src["n"]))]
for L in loci:
    for k in ("K", "gamma", "sharing_param"):
        L[k] = float(L[k])
B = P.LocusBatch(loci, int(src["c"]), search=True)
B.buf.fill(np.nan)
B.run()
np.savez(sys.argv[3], buf=B.buf, cnt=B.cnt, it=B.iterations, why=B.stop_reasons)
"""


@pytest.mark.parametrize("threads", [1, 2, 8])
def test_other_thread_counts(threads, tmp_path):
    import pipsort_b200 as P
    D = [as_dict(L) for L in loci()]
    src, dst = tmp_path / "loci.npz", tmp_path / "results.npz"
    np.savez(src, n=len(D), c=5, **{f"{k}{i}": v for i, L in enumerate(D) for k, v in L.items()})
    env = dict(os.environ, PIPSORT_BATCH_THREADS=str(threads))
    p = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(src), str(dst)], capture_output=True, text=True, env=env,
                       timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    B = P.LocusBatch(D, 5, search=True)
    out = np.load(dst)
    B.buf[:] = out["buf"]                                   # the same layout: slice the child's buffer as this one
    B.cnt[:] = out["cnt"]
    check_against_one_at_a_time((B.results(), out["it"], out["why"]), 5)


# ---- 3. failures inside a batch -----------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def singular_search_locus():
    """make_locus(12, overlap=0.5, seed=41) with Sigma_0[i][j] = 1.5 for the SNP the search moves to in round 0 and another
    SNP of study 0: round 0 scores single SNPs only, which the off-diagonal entry does not change, so the search still moves
    there, and round 1 scores the pair (its plus group) -- an indefinite 2x2 block, as test_gpu_batch's singular_locus."""
    from oracle import oracle as O
    from pipsort_b200 import synth
    SL = synth.make_locus(12, overlap=0.5, seed=41)
    U, smap = SL.snp_map.shape[1], SL.snp_map
    want = O.sss(as_oracle(SL), 3)
    a = S.states(U, 3, want.extra["trace"])[1][0]
    b = next(h for h in range(U) if h != a and smap[0, h] >= 0)
    i, j = int(smap[0, a]), int(smap[0, b])
    sig0 = np.array(SL.sigma[0])
    sig0[i, j] = sig0[j, i] = 1.5
    assert want.extra["n_iter"] >= 2 and float(SL.d[0]) > 20
    return dataclasses.replace(SL, sigma=[sig0, SL.sigma[1]])


def bad_locus(kind):
    base = loci()[17]
    if kind == "p1":
        return as_dict(base, sharing_param=1.0)
    if kind == "U":                          # 32767 union SNPs that neither study has: refused before any engine exists
        U = S_MAX_U + 1
        return dict(num_snps=np.zeros(2, dtype=np.int32), sigma=np.zeros(0), z=np.zeros(0), d=np.array([5.72, 5.72]), K=0.0,
                    snp_map=np.full((2, U), -1, dtype=np.int32), gamma=0.01, sharing_param=0.75)
    return as_dict(singular_search_locus())


S_MAX_U = (1 << 15) - 2
FAILURES = {"p1": (PIPSORT_E_ARG, "locus 17: the shotgun search is undefined at sharing_param = 1"),
            "U": (PIPSORT_E_RANGE, "locus 17: the search state packs union indices into 15 bits"),
            "singular": (PIPSORT_E_SINGULAR, "matrix is singular")}


@pytest.mark.parametrize("kind", list(FAILURES))
def test_failure_inside_a_batch(kind, pool_used):  # noqa: F811
    import pipsort_b200 as P
    code, text = FAILURES[kind]
    if kind == "singular":                    # one-at-a-time pipsort_sss reports it too
        with engine_for(singular_search_locus(), 3) as e:
            expect_error(code, text, e.sss, 3)
    good = P.LocusBatch([as_dict(L) for L in loci()], 3, search=True)
    run_fresh(good)                           # warm-up: the streams, events and pinned staging of the engines in flight
    base = pool_used()
    D = [as_dict(L) for L in loci()]
    D[17] = bad_locus(kind)
    expect_error(code, text, run_fresh, P.LocusBatch(D, 3, search=True))
    assert text in P.lib().pipsort_last_error().decode()
    assert pool_used() == base
    check_against_one_at_a_time(run_fresh(good), 3)
