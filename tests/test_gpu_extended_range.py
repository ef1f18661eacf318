"""The exhaustive, scoring and explicit-configuration paths beyond the plain-double range and above c = 3, against the oracle.

* Class 3 on loci that leave the register kernel's fast range in every way it can be left (range_loci.py: strong single
  SNPs, pairs and triples beyond 2^450, in both studies, as a, b and x, next to fast lanes of the same warp-step) and on
  one that sits right at the limits; the tests/example locus at c = 3 (real data, ~80 exponent bins per accumulator).
* The warp-per-configuration kernel of the classes above 3 (c = 4 .. 8), alone and together with the register kernel.
* Scoring batches with up to 8 SNPs per row, the shotgun search and explicit configurations on the strong locus.
* Sharing parameters at the edges: p = 1e-9, 0.999999 and 1.

Besides assert_results_match (1e-10 relative), every log-space value must agree with the oracle to 1e-8 nats absolute:
the results here are up to a few thousand nats in magnitude, so that bound is tighter than the relative one.
"""
import dataclasses
import functools
import itertools
from math import comb

import numpy as np
import pytest

import range_loci as R
from conftest import assert_results_match, engine_for, exh_plan_env, oracle_locus, synth_as_oracle_locus

pytestmark = pytest.mark.gpu

ATOL_NATS = 1e-8
PRIOR_WEIGHTED = ("total", "post", "noCausal", "sharedPips")     # the rest (sharedLL, notSharedLL) carry no prior


def _arrays(r):
    post = getattr(r, "postValues", None)
    return {"total": np.array([r.total]), "post": np.asarray(r.post if post is None else post),
            "noCausal": np.asarray(r.noCausal), "sharedPips": np.asarray(r.sharedPips),
            "sharedLL": np.asarray(r.sharedLL), "notSharedLL": np.asarray(r.notSharedLL)}


def _with(want, arrays):
    from oracle import oracle as O
    return O.Result(float(arrays["total"][0]), arrays["post"], arrays["noCausal"], arrays["sharedPips"], arrays["sharedLL"],
                    arrays["notSharedLL"], getattr(want, "n_eval", 0))


def check(got, want, n_configs=None, zero_prior=False, atol_nc=ATOL_NATS):
    """assert_results_match + every log-space value within ATOL_NATS of the oracle.  zero_prior (p = 1): the oracle, like
    the reference's addlogSpace, returns -inf for a prior-weighted accumulator whose every contribution has prior 0; the
    engine returns 0.0 ("empty") there.  PIPs and the output files are the same either way (exp(-inf - total) = 0 and an
    empty accumulator is reported as 0), so for those arrays -inf is read as 0.0; the likelihood-only arrays must agree as
    they are."""
    w = _arrays(want)
    if zero_prior:
        for k in PRIOR_WEIGHTED:
            w[k] = np.where(np.isneginf(w[k]), 0.0, w[k])
        want = _with(want, w)
    for k, v in w.items():
        assert np.all(np.isfinite(v)), f"{k}: oracle value not finite"
    if n_configs is not None:
        assert got.n_configs == n_configs
    assert_results_match(got, want)
    g = _arrays(got)
    for k in w:
        np.testing.assert_allclose(g[k], w[k], rtol=0, atol=atol_nc if k == "noCausal" else ATOL_NATS, err_msg=k)
    print("largest log-space difference: %.3e nats" % max(float(np.max(np.abs(g[k] - w[k]), initial=0.0)) for k in w))


# ---- loci and oracle results, once per session --------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def straddle(p=0.75):
    return dataclasses.replace(R.straddle_locus(), sharing_param=p)


@functools.lru_cache(maxsize=None)
def threshold():
    return R.threshold_locus()[0]


@functools.lru_cache(maxsize=None)
def fast30():
    from pipsort_b200 import synth
    return synth.make_locus(20, overlap=0.5, seed=303)          # U = 30, everything in the fast range


@functools.lru_cache(maxsize=None)
def synth12():
    from pipsort_b200 import synth
    return synth.make_locus(8, overlap=0.5, seed=12)            # U = 12


@functools.lru_cache(maxsize=None)
def lone():
    return R.lone_strong_locus()


@functools.lru_cache(maxsize=None)
def spread():
    return R.spread_locus()


LOCI = {"straddle": straddle, "threshold": threshold, "fast30": fast30, "synth12": synth12, "lone": lone, "spread": spread}


def locus(name, p=None):
    if name == "small_example":
        return oracle_locus("small_example")
    if name == "straddle" and p is not None:
        return straddle(p)
    return LOCI[name]()


@functools.lru_cache(maxsize=None)
def oracle_exh(name, c, lo=0, hi=None, p=None):
    from oracle import oracle as O
    L = locus(name, p)
    OL = L if name == "small_example" else synth_as_oracle_locus(L)
    if hi is None:
        hi = O.total_union_subsets(OL.U, c)
    return O.exhaustive_omp_full(OL, c, lo, hi)


def n_configs(name, c):
    from pipsort_b200 import synth
    return synth.count_configs(locus(name).snp_map, c)


def class_offset(U, j):
    return sum(comb(U, i) for i in range(j))


def rank3(U, a, b, x):
    """Rank of the triple a < b < x (snp_map order) in the rank space of c >= 3."""
    r = class_offset(U, 3)
    for i in range(a):
        r += comb(U - 1 - i, 2)
    for i in range(a + 1, b):
        r += U - 1 - i
    return r + (x - b - 1)


def strong_snps(L):
    """Union positions of the SNPs with a slow single in either study, in snp_map order."""
    out = set()
    for s in range(2):
        slow = R.e1n(L, s) >= R.E1_LIMIT
        out |= {int(g) for g in np.nonzero(L.snp_map[s] >= 0)[0] if slow[L.snp_map[s, g]]}
    return sorted(out)


# ---- 1. class 3 on the straddle locus -----------------------------------------------------------------------------------
@pytest.mark.parametrize("keep_order,generic_only", [(False, False), (True, False), (False, True)])
def test_straddle_c3_whole(keep_order, generic_only):
    L = straddle()
    with engine_for(L, 3, keep_order=keep_order, generic_only=generic_only) as e:
        r = e.compute_total_likelihood(3)
    check(r, oracle_exh("straddle", 3), n_configs("straddle", 3))


def straddle_ranges():
    L = straddle()
    U = L.U
    st = strong_snps(L)
    g1, g2 = st[0], st[len(st) // 2]
    first = lambda a: rank3(U, a, a + 1, a + 2)              # noqa: E731
    tot = class_offset(U, 4)
    return [(first(g1) + 5, first(g1 + 3) + 2),             # starts inside the a of a strong SNP
            (first(g2) - 40, first(g2) + 9),                # ends inside the a of a strong SNP
            (class_offset(U, 3) - 100, class_offset(U, 3) + 100),   # across the 2 -> 3 class boundary
            (tot - 500, tot)]                               # the end


@pytest.mark.parametrize("chunk", [None, 1, 7, 40])
def test_straddle_c3_partial_ranges(chunk):
    """Partial rank ranges (the reference's rank space: snp_map order) under forced work decompositions."""
    L = straddle()
    with engine_for(L, 3, keep_order=True) as e, exh_plan_env(chunk):
        for lo, hi in straddle_ranges():
            e.reset()
            e.run_exhaustive(3, lo, hi)
            want = oracle_exh("straddle", 3, lo, hi)
            check(e.read(), want, want.n_eval)


@pytest.mark.parametrize("parts", [2, 3, 8])
def test_straddle_c3_shards_merge(parts):
    L = straddle()
    engines = [engine_for(L, 3) for _ in range(parts)]
    try:
        b = engines[0].shard_ranks(3, parts)
        assert b[0] == 0 and b[-1] == engines[0].total_ranks(3)
        for i, e in enumerate(engines):
            e.run_exhaustive(3, b[i], b[i + 1])
        for e in engines[1:]:
            engines[0].merge_from(e)
        check(engines[0].read(), oracle_exh("straddle", 3), n_configs("straddle", 3))
    finally:
        for e in engines:
            e.close()


# ---- 2. the limits ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("keep_order", [False, True])
def test_threshold_c3(keep_order):
    with engine_for(threshold(), 3, keep_order=keep_order) as e:
        r = e.compute_total_likelihood(3)
    check(r, oracle_exh("threshold", 3), n_configs("threshold", 3))


@pytest.mark.parametrize("keep_order", [False, True])
def test_lone_strong_snp_c3(keep_order):
    """One strong SNP of study 0 only: the triples in which it is a and b, x are of study 1 only take the slow path because
    of a alone, and they dominate the cells of those b and x."""
    with engine_for(lone(), 3, keep_order=keep_order) as e:
        r = e.compute_total_likelihood(3)
    check(r, oracle_exh("lone", 3), n_configs("lone", 3))


# ---- 3. tests/example at c = 3 ------------------------------------------------------------------------------------------
def test_example_c3():
    """47 M configurations; study 0 has 258 pairs beyond 2^450 (~80 bins per accumulator: the scanning finalize)."""
    from oracle import oracle as O
    L = oracle_locus("example", p=0.25)
    want = O.exhaustive_omp_full(L, 3)
    with engine_for(L, 3) as e:
        r = e.compute_total_likelihood(3)
    # each noCausal accumulator of the oracle takes ~4.7e7 log-space additions, each rounded to ulp(4.3e4 nats) = 7e-12: its
    # own result moves by up to 1.1e-8 nats between 3, 8 and 16 threads (the engine sums in linear space and takes one log)
    check(r, want, want.n_eval, atol_nc=5e-8)


# ---- 4. above c = 3: the generic kernel ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name,c", [("straddle", 4), ("fast30", 5)])
@pytest.mark.parametrize("keep_order", [False, True])
def test_generic_classes(name, c, keep_order):
    """straddle at c = 4: C(60,4) = 487,635 subsets of class 4 (the 16-subset chunks of the generic launch)."""
    with engine_for(locus(name), c, keep_order=keep_order) as e:
        r = e.compute_total_likelihood(c)
    check(r, oracle_exh(name, c), n_configs(name, c))


def test_straddle_c4_partial_ranges_across_3_to_4():
    """Ranges that end in class 3 (register kernel) and continue in class 4 (generic kernel) in one call."""
    L = straddle()
    off4 = class_offset(L.U, 4)
    with engine_for(L, 4, keep_order=True) as e:
        for lo, hi in [(off4 - 3000, off4 + 5000), (rank3(L.U, 20, 30, 40), off4 + 100000), (off4 - 1, off4 + 1)]:
            e.reset()
            e.run_exhaustive(4, lo, hi)
            want = oracle_exh("straddle", 4, lo, hi)
            check(e.read(), want, want.n_eval)


def test_straddle_c4_shards_merge():
    L = straddle()
    engines = [engine_for(L, 4) for _ in range(4)]
    try:
        b = engines[0].shard_ranks(4, 4)
        for i, e in enumerate(engines):
            e.run_exhaustive(4, b[i], b[i + 1])
        for e in engines[1:]:
            engines[0].merge_from(e)
        check(engines[0].read(), oracle_exh("straddle", 4), n_configs("straddle", 4))
    finally:
        for e in engines:
            e.close()


@pytest.mark.parametrize("name", ["small_example", "synth12"])
def test_every_class_up_to_8(name):
    L = locus(name)
    with engine_for(L, 8) as e:
        for c in range(9):
            r = e.compute_total_likelihood(c)
            want = oracle_exh(name, c)
            check(r, want, want.n_eval)


def test_wide_exponent_spread_generic_and_batch():
    """d of study 0 ~ 10^12: the expansions of one configuration span up to 2^160 (1/sqrt(A) per study-0 SNP, A ~ 10^12).
    Exhaustive c = 7 (generic kernel for classes 4..7) and a batch of 6-8 SNPs per row."""
    from oracle import oracle as O
    L = spread()
    want = oracle_exh("spread", 7)
    rng = np.random.default_rng(8)
    idx = np.full((48, 8), -1, dtype=np.int32)
    for i in range(len(idx)):
        k = int(rng.integers(6, 9))
        idx[i, :k] = np.sort(rng.choice(L.U, k, replace=False))
    want_l, want_b = O.score_union_configs(synth_as_oracle_locus(L), idx)
    with engine_for(L, 8) as e:
        check(e.compute_total_likelihood(7), want, want.n_eval)
        e.reset()
        got_l = e.score_union_configs(idx)
        np.testing.assert_allclose(got_l, want_l, rtol=0, atol=ATOL_NATS)
        check(e.read(), want_b)


# ---- 5. scoring batches, the shotgun search ------------------------------------------------------------------------------
def strong_rows(rng, L, n, kmax):
    """n rows of up to kmax union SNPs (-1 padded); most contain at least one strong SNP."""
    st = strong_snps(L)
    idx = np.full((n, kmax), -1, dtype=np.int32)
    for i in range(n):
        k = int(rng.integers(0 if i == 0 else 1, kmax + 1))
        pick = set(rng.choice(L.U, k, replace=False).tolist())
        if k and i % 4:
            pick.pop()
            pick.add(int(rng.choice([g for g in st if g not in pick])))
        idx[i, :len(pick)] = sorted(pick)
    return idx


def _score_check(L, kmax, seed, zero_prior=False):
    from oracle import oracle as O
    rng = np.random.default_rng(seed)
    OL = synth_as_oracle_locus(L)
    idx = strong_rows(rng, L, 96, kmax)
    upd = (rng.uniform(size=len(idx)) < 0.7).astype(np.uint8)
    want_l, want = O.score_union_configs(OL, idx, upd)
    idx2 = strong_rows(rng, L, 41, kmax)
    want_l2, want2 = O.score_union_configs(OL, idx2, None, want)
    with engine_for(L, max(kmax, 3)) as e:
        got_l = e.score_union_configs(idx, upd)
        np.testing.assert_allclose(got_l, want_l, rtol=1e-10, atol=0)
        np.testing.assert_allclose(got_l, want_l, rtol=0, atol=ATOL_NATS)
        check(e.read(), want, zero_prior=zero_prior)
        got_l2 = e.score_union_configs(idx2)
        np.testing.assert_allclose(got_l2, want_l2, rtol=0, atol=ATOL_NATS)
        check(e.read(), want2, zero_prior=zero_prior)


@pytest.mark.parametrize("kmax", [3, 5, 8])
def test_straddle_scoring_batches(kmax):
    _score_check(straddle(), kmax, 100 + kmax)


def test_straddle_sss():
    from oracle import oracle as O
    L = straddle()
    want = O.sss(synth_as_oracle_locus(L), 3, max_iter=40)
    with engine_for(L, 3) as e:
        r, iters, why = e.sss(3, max_iterations=40)
    assert iters == want.extra["n_iter"]
    assert why in ((0,) if iters == 40 else (1, 2))
    check(r, want)


# ---- 6. explicit configurations ------------------------------------------------------------------------------------------
def test_straddle_given_configs():
    from oracle import oracle as O
    L = straddle()
    rng = np.random.default_rng(6)
    # global SNP indices (study 0, then study 1), up to 8 per row, most rows with a strong SNP
    strong = [int(L.snp_map[s, g]) + s * int(L.num_snps[0]) for g in strong_snps(L) for s in range(2) if L.snp_map[s, g] >= 0]
    M = np.full((2000, 9), -1, dtype=np.int16)
    for r in range(len(M)):
        k = int(rng.integers(0, 9))
        pick = set(rng.choice(L.N, size=k, replace=False).tolist())
        if k and r % 3:
            pick.pop()
            pick.add(int(rng.choice([g for g in strong if g not in pick])))
        M[r, np.sort(rng.choice(9, size=len(pick), replace=False))] = sorted(pick)
    rc, want = O.given_configs(synth_as_oracle_locus(L), M)
    assert rc == 0
    with engine_for(L, 3) as e:
        r = e.compute_total_likelihood_given_configs(M)
    check(r, want, len(M))


# ---- 7. sharing parameters at the edges ----------------------------------------------------------------------------------
@pytest.mark.parametrize("p", [1e-9, 0.999999, 1.0])
def test_extreme_sharing_exhaustive(p):
    L = straddle(p)
    with engine_for(L, 3) as e:
        r = e.compute_total_likelihood(3)
    check(r, oracle_exh("straddle", 3, p=p), n_configs("straddle", 3), zero_prior=(p == 1.0))


@pytest.mark.parametrize("p", [1e-9, 0.999999, 1.0])
def test_extreme_sharing_batch(p):
    _score_check(straddle(p), 5, 7, zero_prior=(p == 1.0))
