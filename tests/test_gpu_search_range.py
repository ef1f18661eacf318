"""The shotgun search and its two scoring kernels at every max_causal up to 8 and across the prior range, against the oracle.

* Whole searches on the flat loci of search_loci.py, which climb to states of max_causal SNPs: c = 0 .. 8, so that the
  searches with c >= 6 score their neighbourhoods on score_batch_kernel (batch length read on the device), p = 0, the
  reference's round-100 convergence rule without any override, an iteration cap inside such a search, and the refusal
  of a search at p = 1.
* The c = 6 round-100 search split over two ranks (the warp kernel's null row without updates on rank 1, the running
  total read at the reference's own round).
* The lane kernel (score_lane.cuh, <= 5 SNPs) and the warp kernel (score.cuh) on identical rows.
* Scoring batches across the prior range, at both sides of the lane kernel's admission test, and at a prior where the
  lane kernel's factorised weights overflow although every table entry is inside its fast range.
"""
import dataclasses
import functools
import itertools
import os
import sys
import tempfile

import numpy as np
import pytest

import range_loci as R
import search_loci as S
from conftest import ROOT, assert_results_match, engine_for, synth_as_oracle_locus

pytestmark = pytest.mark.gpu

PRIOR_WEIGHTED = ("post", "noCausal", "sharedPips")


def _zero_prior(want):
    """At p = 1 the oracle returns -inf for a prior-weighted accumulator whose every term has prior 0; the engine returns
    0.0 ("empty"): the same PIPs and output files (test_gpu_extended_range.py)."""
    from oracle import oracle as O
    f = {k: np.where(np.isneginf(getattr(want, k)), 0.0, getattr(want, k)) for k in PRIOR_WEIGHTED}
    return O.Result(want.total, f["post"], f["noCausal"], f["sharedPips"], want.sharedLL, want.notSharedLL)


@functools.lru_cache(maxsize=None)
def oracle_search(name, max_iter=1000):
    from oracle import oracle as O
    SL, c = S.search_locus(name)
    return O.sss(synth_as_oracle_locus(SL), c, max_iter=max_iter)


# ---- 1. whole searches ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,engine_c", [(n, S.SEARCHES[n][2]) for n in sorted(S.SEARCHES) if S.SEARCHES[n][2] > 0]
                         + [("c0", 8), ("c5", 8), ("p0_c4", 8)])
def test_search_matches_oracle(name, engine_c):
    """Rounds, stop reason and every accumulator of the whole search equal the oracle's, on an engine created with
    max_causal = c or 8.  The round-100 cases stop by the reference's convergence rule with no environment override."""
    SL, c = S.search_locus(name)
    want = oracle_search(name)
    with engine_for(SL, engine_c) as e:
        r, iters, why = e.sss(c)
    assert (iters, why) == (want.extra["n_iter"], S.stop_reason(want))
    assert (iters, why) == S.SEARCHES[name][3:]
    assert_results_match(r, want)


def test_search_capped_inside_a_round_100_search():
    SL, c = S.search_locus("c7_round100")
    want = oracle_search("c7_round100", 60)
    with engine_for(SL, c) as e:
        r, iters, why = e.sss(c, max_iterations=60)
        assert (iters, why) == (60, 0)
        assert_results_match(r, want)
        r, iters, why = e.sss(c)                       # the same engine runs the whole search afterwards
    assert (iters, why) == (100, 2)
    assert_results_match(r, oracle_search("c7_round100"))


def test_search_refused_at_p1():
    """At p = 1 every neighbour's largest-|l| value is -inf (test_search_loci_cpu.py): the search is refused with
    PIPSORT_E_ARG, and the engine stays usable."""
    import pipsort_b200 as P
    from oracle import oracle as O
    SL, _ = S.search_locus("p0_c4")
    SL = S.with_prior(SL, p=1.0)
    with engine_for(SL, 4) as e:
        with pytest.raises(P.PipsortError) as ei:
            e.sss(4)
        assert ei.value.code == 1
        r, iters, why = e.sss(0)                       # c = 0 draws nothing: the null configuration, then the break
        assert (iters, why) == (0, 1)
        want = O.sss(synth_as_oracle_locus(SL), 0)
        assert_results_match(r, want)


# ---- 2. split search ------------------------------------------------------------------------------------------------
def _split_worker(rank, world, initfile, outdir):
    import faulthandler
    faulthandler.dump_traceback_later(240, exit=True)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    import torch.distributed as dist
    from pipsort_b200 import distributed as D
    dist.init_process_group("gloo", init_method=f"file://{initfile}", rank=rank, world_size=world)
    try:
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        SL, c = S.search_locus("c6_round100")
        with engine_for(SL, c, device=dev) as e:
            one, it1, why1 = e.sss(c)
            assert (it1, why1) == (100, 2)
            assert D.connect_p2p(e)
            r, iters, why = D.sss_sharded(e, c)
            assert (iters, why) == (it1, why1)
            if rank == 0:
                assert_results_match(r, one, rtol=1e-12)
                assert_results_match(r, oracle_search("c6_round100"))
            else:
                assert r is None
        open(os.path.join(outdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_split_search_c6_round_100():
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_split_worker, args=(2, os.path.join(tmp, "init"), tmp), nprocs=2, join=True)
        assert all(os.path.exists(os.path.join(tmp, f"ok{r}")) for r in range(2))


# ---- 3. lane kernel against warp kernel ---------------------------------------------------------------------------------
def _types(SL):
    smap = np.asarray(SL.snp_map)
    return np.where((smap[0] >= 0) & (smap[1] >= 0), 0, np.where(smap[0] >= 0, 1, 2))


def mixed_rows(SL, seed, kmax=5, per_k=48):
    """The null row, then per_k rows of each size 1..kmax (sorted by size: whole warp-steps of 1 and of 2 SNPs), with every
    SNP type (both studies / study 0 only / study 1 only) at every position of every size."""
    rng = np.random.default_rng(seed)
    t = _types(SL)
    rows = [[]]
    for k in range(1, kmax + 1):
        want = {(i, ty) for i in range(k) for ty in range(3)}
        got, mine = set(), []
        while len(mine) < per_k or not want <= got:
            v = sorted(rng.choice(SL.U, k, replace=False).tolist())
            new = {(i, int(t[g])) for i, g in enumerate(v)} - got
            if len(mine) < per_k or new:
                mine.append(v)
                got |= new
        rows += mine
    idx = np.full((len(rows), kmax), -1, dtype=np.int32)
    for i, v in enumerate(rows):
        idx[i, :len(v)] = v
    return idx


@functools.lru_cache(maxsize=None)
def straddle():
    return R.straddle_locus()


@pytest.mark.parametrize("which", ["flat", "straddle"])
def test_lane_and_warp_kernels_on_identical_rows(which):
    """One batch as a 5-column matrix (lane kernel) and again with a sixth, all -1 column (warp kernel): both against the
    oracle, and against each other to 1e-12.  The straddle locus adds rows outside the plain-double range."""
    from oracle import oracle as O
    SL = S.search_locus("c5")[0] if which == "flat" else straddle()
    assert S.lane_ok(SL.gamma, SL.sharing_param)
    idx5 = mixed_rows(SL, 11)
    idx6 = np.concatenate([idx5, np.full((len(idx5), 1), -1, dtype=np.int32)], axis=1)
    rng = np.random.default_rng(12)
    upd = (rng.uniform(size=len(idx5)) < 0.75).astype(np.uint8)
    upd[0] = 1
    want_l, want = O.score_union_configs(synth_as_oracle_locus(SL), idx5, upd)
    with engine_for(SL, 6) as e:
        lane_l = e.score_union_configs(idx5, upd)
        lane = e.read()
        e.reset()
        warp_l = e.score_union_configs(idx6, upd)
        warp = e.read()
    for got_l, got in ((lane_l, lane), (warp_l, warp)):
        np.testing.assert_allclose(got_l, want_l, rtol=1e-10, atol=0)
        assert_results_match(got, want)
        assert got.n_configs == lane.n_configs
    np.testing.assert_allclose(lane_l, warp_l, rtol=1e-12, atol=0)
    assert_results_match(lane, warp, rtol=1e-12)


# ---- 4. the prior range ----------------------------------------------------------------------------------------------
def sized_rows(rng, U, n, kmax):
    """n rows sorted by size: the null row, then sizes drawn from 1..kmax."""
    ks = np.sort(np.concatenate([[0], rng.integers(1, kmax + 1, n - 1)]))
    idx = np.full((n, kmax), -1, dtype=np.int32)
    for i, k in enumerate(ks):
        idx[i, :k] = np.sort(rng.choice(U, int(k), replace=False))
    return idx


def _score_against_oracle(SL, kmax, seed, n=80):
    from oracle import oracle as O
    rng = np.random.default_rng(seed)
    idx = sized_rows(rng, SL.U, n, kmax)
    upd = (rng.uniform(size=n) < 0.8).astype(np.uint8)
    want_l, want = O.score_union_configs(synth_as_oracle_locus(SL), idx, upd)
    with engine_for(SL, max(kmax, 3)) as e:
        got_l = e.score_union_configs(idx, upd)
        got = e.read()
    np.testing.assert_allclose(got_l, want_l, rtol=1e-10, atol=0)
    assert_results_match(got, _zero_prior(want) if SL.sharing_param == 1.0 else want)


@pytest.mark.parametrize("kmax", [3, 5, 8])
@pytest.mark.parametrize("gamma", [1e-6, 0.01, 0.5])
@pytest.mark.parametrize("p", [0.0, 1e-9, 0.2, 1 / 3, 0.75, 0.999999, 1.0])
def test_scoring_across_priors(p, gamma, kmax):
    SL = S.with_prior(S.search_locus("c5")[0], gamma=gamma, p=p)
    _score_against_oracle(SL, kmax, 1000 + kmax)


@pytest.mark.parametrize("p", [1e-38, 1e-40])
@pytest.mark.parametrize("gamma", [0.01, 0.5])
def test_scoring_at_the_lane_admission_boundary(p, gamma):
    """rho^8 a normal double at p = 1e-38 (lane kernel), not at 1e-40 (warp kernel)."""
    assert S.lane_ok(gamma, p) == (p == 1e-38)
    SL = S.with_prior(S.search_locus("c5")[0], gamma=gamma, p=p)
    _score_against_oracle(SL, 5, 7)


def overflow_locus():
    """The c5 flat locus with one shared SNP at log2 E_0({i}) = 449.99, outside every LD block of study 0, under gamma =
    0.99999 and p = 2e-39: rho^8 is a normal double, yet w0[1] E = pi'(5, 0) rho^-4 E overflows in the lane kernel.
    Returns (locus, i as a union index)."""
    SL = S.search_locus("c5")[0]
    g = int(np.nonzero(_types(SL) == 0)[0][0])
    i = int(SL.snp_map[0, g])
    sig0 = np.array(SL.sigma[0])
    sig0[i, :] = 0.0
    sig0[:, i] = 0.0
    sig0[i, i] = 1.0
    SL = dataclasses.replace(SL, sigma=[sig0, SL.sigma[1]])
    z = [np.array(v) for v in SL.z]
    z[0][i] = R.z_for_bits(SL, 0, i, 449.99)
    SL = dataclasses.replace(SL, z=z)
    SL = dataclasses.replace(SL, K=R.choose_K(SL))
    return S.with_prior(SL, gamma=0.99999, p=2e-39), g


def test_lane_weight_overflow_goes_to_the_warp_kernel():
    """Rows of five SNPs holding the strong SNP, every sub-mask of both studies inside the fast range (< 2^450, checked
    with range_loci.log2_e): the oracle's values are finite, and so must the engine's be."""
    from oracle import oracle as O
    SL, g = overflow_locus()
    assert S.lane_ok_rho_only(SL.sharing_param) and not S.lane_ok(SL.gamma, SL.sharing_param)
    rng = np.random.default_rng(21)
    others = [u for u in range(SL.U) if u != g]
    rows, top = [], -np.inf
    while len(rows) < 40:
        v = sorted([g] + rng.choice(others, 4, replace=False).tolist())
        worst = -np.inf
        for s in range(2):
            loc = [int(SL.snp_map[s, u]) for u in v if SL.snp_map[s, u] >= 0]
            for r in range(1, len(loc) + 1):
                worst = max(worst, float(np.max(R.log2_e(SL, s, np.array(list(itertools.combinations(loc, r)))))))
        if worst < S.FAST_BITS:
            rows.append(v)
            top = max(top, worst)
    assert top > 449.9
    idx = np.array(rows, dtype=np.int32)
    want_l, want = O.score_union_configs(synth_as_oracle_locus(SL), idx)
    assert np.all(np.isfinite(want_l)) and np.isfinite(want.total)
    with engine_for(SL, 5) as e:
        got_l = e.score_union_configs(idx)
        got = e.read()
    np.testing.assert_allclose(got_l, want_l, rtol=1e-10, atol=0)
    assert_results_match(got, want)
