"""One exhaustive pass, a grid of priors: engines created with prior_classes=True (PIPSORT_PRIOR_CLASSES) keep the
accumulators unweighted per prior class and apply any number of priors (gamma, p) when the results are read.

Every prior of a grid must give what an engine created with that prior gives: the reference dumps, the oracle run per prior,
and ordinary engines (same n_configs, same empty pattern -- p = 1 included), on the register kernel's fast and slow paths, the
generic kernel, partial rank ranges and merged shards.
"""
import functools
import itertools

import numpy as np
import pytest

import range_loci as R
from conftest import (args_to_params, assert_results_match, engine_for, exh_plan_env, golden, has_golden, oracle_locus,
                      synth_as_oracle_locus, synth_locus)

pytestmark = pytest.mark.gpu

GAMMAS = (1e-3, 0.01, 0.2)
PS = (0.0, 1e-9, 0.25, 0.75, 0.999999, 1.0)
GRID = list(itertools.product(GAMMAS, PS))
SMALL_GRID = [(0.01, 0.0), (0.01, 0.75), (1e-3, 1.0), (0.2, 0.25), (0.01, 1e-9)]


def with_prior(L, gamma, p):
    import copy
    import dataclasses
    key = "sharing_param" if hasattr(L, "sharing_param") else "p"
    if dataclasses.is_dataclass(L):
        return dataclasses.replace(L, gamma=gamma, **{key: p})
    L2 = copy.copy(L)
    L2.gamma = gamma
    setattr(L2, key, p)
    return L2


def ordinary(L, c, gamma, p, **kw):
    """Results of an engine created with the prior (gamma, p) after a whole pass."""
    with engine_for(with_prior(L, gamma, p), c, **kw) as e:
        return e.compute_total_likelihood(c)


def grid_pass(L, c, priors, runs=None, **kw):
    """One class-resolved engine, one pass (or the given rank ranges), the grid read."""
    with engine_for(L, c, prior_classes=True, **kw) as e:
        e.reset()
        for lo, hi in (runs or [(0, None)]):
            e.run_exhaustive(c, lo, hi)
        return e.read_prior_grid(priors)


def same(got, want):
    assert got.n_configs == want.n_configs
    assert_results_match(got, want)


def match_oracle(got, want):
    """assert_results_match against the oracle; its -inf (every contribution of prior 0, p = 1) is the engine's 0.0."""
    from oracle import oracle as O
    fix = lambda a: np.where(np.isneginf(a), 0.0, a)     # noqa: E731
    w = O.Result(0.0 if np.isneginf(want.total) else want.total, fix(np.asarray(want.post)), fix(np.asarray(want.noCausal)),
                 fix(np.asarray(want.sharedPips)), np.asarray(want.sharedLL), np.asarray(want.notSharedLL), want.n_eval)
    assert got.n_configs == want.n_eval
    assert_results_match(got, w)


# ---- 1. reference dumps: goldens that share (dataset, c, s, t) from ONE engine ---------------------------------------------
@pytest.mark.parametrize("keep_order", [False, True])
@pytest.mark.parametrize("names", [("small_c3_p075", "small_c3_p0"), ("small_c2_p025", "small_c2_p075")])
def test_grid_matches_reference_dumps(names, keep_order):
    if not all(has_golden(n) for n in names):
        pytest.skip("golden not generated")
    gs = [golden(n) for n in names]
    prms = [args_to_params(g["args"]) for g in gs]
    key = {(g["dataset"], p["c"], p["s"], p["t"]) for g, p in zip(gs, prms)}
    assert len(key) == 1
    p0 = prms[0]
    L = oracle_locus(gs[0]["dataset"], p=p0["p"], gamma=p0["gamma"], s=p0["s"], t=p0["t"])
    res = grid_pass(L, p0["c"], [(p["gamma"], p["p"]) for p in prms], keep_order=keep_order)
    for r, g in zip(res, gs):
        assert_results_match(r, g)


@pytest.mark.parametrize("keep_order", [False, True])
def test_grid_example_dump_and_oracle(keep_order):
    from oracle import oracle as O
    if not has_golden("example_c2_p025"):
        pytest.skip("golden not generated")
    g = golden("example_c2_p025")
    prm = args_to_params(g["args"])
    L = oracle_locus(g["dataset"], p=prm["p"], gamma=prm["gamma"], s=prm["s"], t=prm["t"])
    extra = [(0.01, 0.75), (0.2, 0.0), (1e-3, 1.0)]
    res = grid_pass(L, 2, [(prm["gamma"], prm["p"])] + extra, keep_order=keep_order)
    assert_results_match(res[0], g)
    if keep_order:      # the oracle once is enough
        for r, (gam, p) in zip(res[1:], extra):
            match_oracle(r, O.exhaustive_omp_full(with_prior(L, gam, p), 2))


# ---- 2. the oracle over a wide grid ----------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def oracle_grid_locus(c):
    from pipsort_b200 import synth
    return synth.make_locus(50 if c == 2 else 40, overlap=0.6, seed=4040 + c)


@pytest.mark.parametrize("c", [2, 3])
def test_grid_matches_oracle_per_prior(c):
    from oracle import oracle as O
    SL = oracle_grid_locus(c)
    res = grid_pass(SL, c, GRID)
    OL = synth_as_oracle_locus(SL)
    for r, (gam, p) in zip(res, GRID):
        match_oracle(r, O.exhaustive_omp_full(with_prior(OL, gam, p), c))


# ---- 3. the same results as an ordinary engine created with each prior --------------------------------------------------
def test_grid_equals_ordinary_150_c3():
    SL = synth_locus(150)
    res = grid_pass(SL, 3, GRID)
    for r, (gam, p) in zip(res, GRID):
        same(r, ordinary(SL, 3, gam, p))


@pytest.mark.parametrize("name", ["straddle", "lone", "threshold"])
def test_grid_equals_ordinary_slow_path(name):
    L = {"straddle": R.straddle_locus, "lone": R.lone_strong_locus, "threshold": lambda: R.threshold_locus()[0]}[name]()
    for keep in (False, True):
        res = grid_pass(L, 3, SMALL_GRID, keep_order=keep)
        for r, (gam, p) in zip(res, SMALL_GRID):
            same(r, ordinary(L, 3, gam, p, keep_order=keep))


def test_grid_equals_ordinary_generic_only():
    SL = synth_locus(40, overlap=0.5, seed=77)
    res = grid_pass(SL, 3, SMALL_GRID, generic_only=True)
    for r, (gam, p) in zip(res, SMALL_GRID):
        same(r, ordinary(SL, 3, gam, p, generic_only=True))
        same(r, ordinary(SL, 3, gam, p))


@pytest.mark.parametrize("c", [4, 5])
def test_grid_equals_ordinary_above_3(c):
    from pipsort_b200 import synth
    SL = synth.make_locus(8, overlap=0.5, seed=12)
    res = grid_pass(SL, c, SMALL_GRID)
    for r, (gam, p) in zip(res, SMALL_GRID):
        same(r, ordinary(SL, c, gam, p))


def test_own_prior_and_one_call():
    """read() / finalize + fetch on a class-resolved engine report its own prior; the one-call grid equals the engine path."""
    import pipsort_b200 as P
    SL = synth_locus(60, overlap=0.7, seed=5)
    want = ordinary(SL, 3, SL.gamma, SL.sharing_param)
    with engine_for(SL, 3, prior_classes=True) as e:
        got = e.compute_total_likelihood(3)
        e.finalize(reset=True)
        fetched = e.fetch()
        e.run_exhaustive(3)                         # the reset finalize left the store empty
        again = e.read_prior_grid([(SL.gamma, SL.sharing_param)])[0]
    same(got, want)
    same(fetched, want)
    same(again, want)
    one = P.posterior_exhaustive_grid(SL.num_snps, SL.sigma, SL.z, SL.d, SL.K, SL.snp_map, 3, SMALL_GRID)
    for r, (gam, p) in zip(one, SMALL_GRID):
        same(r, ordinary(SL, 3, gam, p))


# ---- 4. partial ranges and shards -------------------------------------------------------------------------------------------
def test_grid_partial_ranges_and_shards():
    SL = synth_locus(40, overlap=0.5, seed=99)
    whole = grid_pass(SL, 3, SMALL_GRID)
    with engine_for(SL, 3) as e:
        total = e.total_ranks(3)
    cuts = [0, 7, 500, 4321, total // 2, total - 3, total]
    for chunk in (None, 1, 7, 40):
        with exh_plan_env(chunk):
            part = grid_pass(SL, 3, SMALL_GRID, runs=list(zip(cuts[:-1], cuts[1:])))
        for a, b in zip(part, whole):
            assert a.n_configs == b.n_configs
            assert_results_match(a, b)
    for parts in (2, 3, 8):
        engines = [engine_for(SL, 3, prior_classes=True) for _ in range(parts)]
        try:
            bounds = engines[0].shard_ranks(3, parts)
            for i, e in enumerate(engines):
                e.reset()
                e.run_exhaustive(3, bounds[i], bounds[i + 1])
            for e in engines[1:]:
                engines[0].merge_from(e)
            merged = engines[0].read_prior_grid(SMALL_GRID)
        finally:
            for e in engines:
                e.close()
        for a, b in zip(merged, whole):
            assert a.n_configs == b.n_configs
            assert_results_match(a, b)


def test_grid_range_across_the_3_to_4_boundary():
    from pipsort_b200 import synth
    from math import comb
    SL = synth.make_locus(8, overlap=0.5, seed=12)
    U = SL.snp_map.shape[1]
    whole = grid_pass(SL, 4, SMALL_GRID)
    b = sum(comb(U, j) for j in range(4))
    part = grid_pass(SL, 4, SMALL_GRID, runs=[(0, b - 17), (b - 17, b + 23), (b + 23, None)])
    for a, w in zip(part, whole):
        assert a.n_configs == w.n_configs
        assert_results_match(a, w)


# ---- 5. refusals ------------------------------------------------------------------------------------------------------------
def test_refusals():
    import pipsort_b200 as P
    SL = synth_locus(20, overlap=0.5, seed=3)
    ARG = 1
    with engine_for(SL, 3, prior_classes=True) as e:
        calls = [lambda: e.sss(3, 5), lambda: e.score_union_configs(np.array([[0, 1]], dtype=np.int32)),
                 lambda: e.score_given_configs(np.array([[0, -1]], dtype=np.int16)),
                 lambda: e.read_prior_grid([]), lambda: e.read_prior_grid([(0.0, 0.5)]), lambda: e.read_prior_grid([(1.0, 0.5)]),
                 lambda: e.read_prior_grid([(0.01, -0.1)]), lambda: e.read_prior_grid([(0.01, 1.5)]),
                 lambda: e.read_prior_grid([(0.01, 0.5), (float("nan"), 0.5)])]
        for f in calls:
            with pytest.raises(P.PipsortError) as ex:
                f()
            assert ex.value.code == ARG
        with pytest.raises(P.PipsortError) as ex:
            e.p2p_combine_finalize()
        assert ex.value.code == ARG
        with pytest.raises(P.PipsortError) as ex:
            e.sss_sharded(3, 5)
        assert ex.value.code == ARG
    with engine_for(SL, 3) as e:
        e.compute_total_likelihood(3)
        with pytest.raises(P.PipsortError) as ex:
            e.read_prior_grid([(0.01, 0.5)])
        assert ex.value.code == ARG
