"""The posterior of the causal counts: engines created with causal_counts=True (PIPSORT_CAUSAL_COUNTS) keep the count table
R[a][b0][b1] beside the class-resolved store, read by Engine.read_count_table / pipsort_count_table_batch.

* The table equals the CPU oracle's (count_oracle.py): the same -inf pattern, finite entries within 1e-10 relative and
  1e-8 nats -- small_example in both SNP orders, tests/example, a mixed-type locus, a locus beyond the plain-double range on
  the register and on the generic kernel, c = 4 and 5 through the generic kernel, and a locus of one SNP per study.
* On the same store it agrees with the existing reads: its log-sum-exp over b0 is read_class_evidence's table (1e-12
  relative), and at every prior of test_gpu_prior_grid.GRID count_posterior gives the grid read's P(k_s = 0), E[a] (shared
  PIPs), E[k_s] (PIPs per study) and total.  The grid read and the class table of a counts engine are a class-resolved
  engine's.  A read that clears the store clears the count table.
* Sums of stores (2 and 3 shards, merged) give the whole pass's table and configuration count.
* The batch equals engine-by-engine tables on 3 and 1 host threads, and stops at a failure at position 17 of 40.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import range_loci as R
from conftest import ROOT, engine_for, oracle_locus, synth_as_oracle_locus, synth_locus
from count_oracle import cnt_classes, count_table
from test_gpu_batch import FAILURES, PIPSORT_E_ARG, as_dict, bad_locus, expect_error, small_loci
from test_gpu_prior_grid import GRID

pytestmark = pytest.mark.gpu


def ncnt(c):
    return (c + 1) * (c + 2) * (c + 3) // 6


def counts_pass(L, c, **kw):
    """One counts engine, one pass: its count table, class table, grid read over GRID, U and n_configs."""
    with engine_for(L, c, causal_counts=True, **kw) as e:
        e.reset()
        e.run_exhaustive(c)
        cnt = e.read_count_table(c)
        tab = e.read_class_evidence(c)
        grid = e.read_prior_grid(GRID)
        return cnt, tab, grid, e.U, e.config_count()


def same_pattern(got, want, rtol=1e-10, atol=1e-8):
    assert not np.isnan(got).any()
    assert np.array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    np.testing.assert_allclose(got[fin], want[fin], rtol=rtol, atol=atol)


# ---- 1. against the oracle --------------------------------------------------------------------------------------------------
def check_oracle(L, c, **kw):
    OL = L if hasattr(L, "n_snps") else synth_as_oracle_locus(L)
    want, n = count_table(OL, c)
    with engine_for(L, max(c, 3), causal_counts=True, **kw) as e:
        e.reset()
        e.run_exhaustive(c)
        got = e.read_count_table(c)
        assert e.config_count() == n
    assert got.shape == (ncnt(c),)
    same_pattern(got, want)
    return got


@pytest.mark.parametrize("keep_order", [False, True])
def test_small_example_c3(keep_order):
    check_oracle(oracle_locus("small_example"), 3, keep_order=keep_order)


def test_example_c2():
    check_oracle(oracle_locus("example", p=0.25), 2)


def test_synthetic_mixed_types():
    check_oracle(synth_locus(30, overlap=0.5, seed=31), 3)


@pytest.mark.parametrize("generic_only", [False, True])
def test_beyond_the_double_range(generic_only):
    check_oracle(R.straddle_locus(), 3, generic_only=generic_only)


@pytest.mark.parametrize("c", [4, 5])
def test_generic_kernel_above_three(c):
    from pipsort_b200 import synth
    check_oracle(synth.make_locus(8, overlap=0.5, seed=500 + c), c)


def one_snp_locus():
    from oracle import oracle as O
    return O.Locus(n_snps=np.array([1, 1], dtype=np.int32), sigma=[np.ones((1, 1)), np.ones((1, 1))],
                   z=[np.array([2.5]), np.array([-1.0])], K=7.25, d=np.array([5.72, 5.72]),
                   snp_map=np.zeros((2, 1), dtype=np.int32), gamma=0.01, p=0.75)


def test_one_snp_per_study():
    """One union SNP in both studies: J = 0 and the three classes of J = 1 hold something, every J >= 2 class is -inf."""
    got = check_oracle(one_snp_locus(), 3)
    assert np.isfinite(got[:4]).all() and np.isneginf(got[4:]).all()


# ---- 2. against the existing reads on the same store -------------------------------------------------------------------------
def check_reads(L, c, **kw):
    import pipsort_b200 as P
    cnt, tab, grid, U, _ = counts_pass(L, c, **kw)
    np.testing.assert_allclose(P.class_tables_from_counts(cnt, c), tab, rtol=1e-12, atol=0)
    assert np.array_equal(np.isneginf(P.class_tables_from_counts(cnt, c)), np.isneginf(tab))
    n0 = L.n_snps[0] if hasattr(L, "n_snps") else L.num_snps[0]
    for (g, p), r in zip(GRID, grid):
        post, ev = P.count_posterior(cnt.reshape(1, -1), [U], g, p)
        q = post[0]
        assert ev[0] == pytest.approx(r.total, rel=1e-12, abs=0), f"gamma={g} p={p}: total"
        assert q.sum() == pytest.approx(1.0, abs=1e-12)
        no = r.no_causal()
        assert q[0, 0, :].sum() == pytest.approx(no[0], abs=1e-8), f"gamma={g} p={p}: P(k0 = 0)"
        assert q[0, :, 0].sum() == pytest.approx(no[1], abs=1e-8), f"gamma={g} p={p}: P(k1 = 0)"
        A, B0, B1 = np.meshgrid(np.arange(c + 1), np.arange(c + 1), np.arange(c + 1), indexing="ij")
        pips = r.pips()
        assert (q * A).sum() == pytest.approx(r.shared_pips().sum(), abs=1e-8), f"gamma={g} p={p}: E[a]"
        assert (q * (A + B0)).sum() == pytest.approx(pips[:n0].sum(), abs=1e-8), f"gamma={g} p={p}: E[k0]"
        assert (q * (A + B1)).sum() == pytest.approx(pips[n0:].sum(), abs=1e-8), f"gamma={g} p={p}: E[k1]"
    return cnt, tab, grid


@pytest.mark.parametrize("name,c", [("small_example", 3), ("example", 2)])
def test_reads_agree(name, c):
    check_reads(oracle_locus(name, p=0.25 if name == "example" else 0.75), c)


def test_reads_agree_synthetic_and_classes_engine():
    SL = synth_locus(30, overlap=0.5, seed=31)
    cnt, tab, grid = check_reads(SL, 3)
    with engine_for(SL, 3, prior_classes=True) as e:
        e.run_exhaustive(3)
        want_tab = e.read_class_evidence(3)
        want_grid = e.read_prior_grid(GRID)
    same_pattern(tab, want_tab, rtol=1e-12, atol=0)
    for got, want in zip(grid, want_grid):
        assert got.total == pytest.approx(want.total, rel=1e-12)
        for k in ("postValues", "noCausal", "sharedPips", "sharedLL", "notSharedLL"):
            a, b = np.asarray(getattr(got, k)), np.asarray(getattr(want, k))
            assert np.array_equal(a == 0.0, b == 0.0), k
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12, err_msg=k)
        assert got.n_configs == want.n_configs


def test_clearing_read_clears_the_count_table():
    """finalize(reset=True) leaves the count table empty: a second pass reads what the first did."""
    SL = synth_locus(20, overlap=0.5, seed=7)
    with engine_for(SL, 3, causal_counts=True) as e:
        e.run_exhaustive(3)
        first = e.read_count_table(3)
        e.finalize(reset=True)
        e.run_exhaustive(3)
        same_pattern(e.read_count_table(3), first, rtol=1e-12, atol=0)


# ---- 3. sums of stores ------------------------------------------------------------------------------------------------------
def test_merged_stores():
    SL = synth_locus(40, overlap=0.5, seed=99)
    whole, _, _, _, n = counts_pass(SL, 3)
    for parts in (2, 3):
        engines = [engine_for(SL, 3, causal_counts=True) for _ in range(parts)]
        try:
            bounds = engines[0].shard_ranks(3, parts)
            for i, e in enumerate(engines):
                e.reset()
                e.run_exhaustive(3, bounds[i], bounds[i + 1])
            for e in engines[1:]:
                engines[0].merge_from(e)
            got = engines[0].read_count_table(3)
            assert engines[0].config_count() == n
        finally:
            for e in engines:
                e.close()
        same_pattern(got, whole)


# ---- 4. batch ---------------------------------------------------------------------------------------------------------------
def one_by_one(D, c):
    import pipsort_b200 as P
    out, cnt = [], []
    for Di in D:
        with P.Engine(Di["num_snps"], Di["sigma"], Di["z"], Di["d"], Di["K"], Di["snp_map"], gamma=Di["gamma"],
                      sharing_param=Di["sharing_param"], max_causal=c, causal_counts=True) as e:
            e.run_exhaustive(c)
            out.append(e.read_count_table(c))
            cnt.append(e.config_count())
    return np.array(out), np.array(cnt, dtype=np.uint64)


def count_batch(D, c):
    import pipsort_b200 as P
    B = P.LocusBatch(D, c, count_table=True)
    B.buf.fill(np.nan)
    B.cnt[:] = 0
    B.run()
    return B.tables(), B.cnt.copy()


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
B = P.LocusBatch(loci, 3, count_table=True)
B.buf.fill(np.nan)
B.cnt[:] = 0
B.run()
np.savez(sys.argv[3], tab=B.tables(), cnt=B.cnt)
"""


def same_tables(got, cnt, want, wcnt):
    assert np.array_equal(cnt, wcnt)
    assert np.array_equal(np.isneginf(got), np.isneginf(want)) and not np.isnan(got).any()
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)


def test_batch_equals_engines(tmp_path):
    import pipsort_b200 as P
    D = [as_dict(L) for L in small_loci()]
    want, wcnt = one_by_one(D, 3)
    same_tables(*count_batch(D, 3), want, wcnt)              # three host threads
    np.testing.assert_allclose(P.class_tables_from_counts(want, 3), P.class_evidence_batch(D, 3), rtol=1e-12, atol=0)
    src, dst = tmp_path / "loci.npz", tmp_path / "tables.npz"
    np.savez(src, n=len(D), **{f"{k}{i}": v for i, L in enumerate(D) for k, v in L.items()})
    env = dict(os.environ, PIPSORT_BATCH_THREADS="1")
    p = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(src), str(dst)], capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    out = np.load(dst)
    same_tables(out["tab"], out["cnt"], want, wcnt)
    assert count_batch([], 3)[0].shape == (0, ncnt(3))


@pytest.mark.parametrize("kind", list(FAILURES))
def test_failure_inside_a_batch(kind):
    D = [as_dict(L) for L in small_loci()]
    want, wcnt = count_batch(D, 3)
    code, text = FAILURES[kind]
    bad = list(D)
    bad[17] = bad_locus(kind)
    expect_error(code, text, count_batch, bad, 3)
    same_tables(*count_batch(D, 3), want, wcnt)


# ---- 5. refusals --------------------------------------------------------------------------------------------------------------
def test_refusals():
    SL = synth_locus(20, overlap=0.5, seed=3)
    for kw in ({}, {"prior_classes": True}):
        with engine_for(SL, 3, **kw) as e:
            e.run_exhaustive(3)
            expect_error(PIPSORT_E_ARG, "PIPSORT_CAUSAL_COUNTS", e.read_count_table, 3)
    with engine_for(SL, 3, causal_counts=True) as e:
        e.run_exhaustive(3)
        expect_error(PIPSORT_E_ARG, "c=4", e.read_count_table, 4)
        expect_error(PIPSORT_E_ARG, "c=-1", e.read_count_table, -1)
        assert np.isfinite(e.read_count_table(3)[0])
        expect_error(PIPSORT_E_ARG, "shotgun search", e.sss, 3)          # (Engine.sss resets the store first)
        expect_error(PIPSORT_E_ARG, "PIPSORT_PRIOR_CLASSES", e.score_union_configs, np.array([[0, -1, -1]], dtype=np.int32))
        expect_error(PIPSORT_E_ARG, "PIPSORT_PRIOR_CLASSES", e.p2p_combine_finalize)
    assert len(cnt_classes(3)) == ncnt(3) == 20 and ncnt(8) == 165
