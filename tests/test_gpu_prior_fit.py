"""Choosing the prior from class tables: Engine.read_class_evidence / pipsort_class_evidence_batch (the table mode of the grid
finalize) and fit_prior (pipsort_fit_prior) on their tables.

* The table of a pass, evaluated at every prior of test_gpu_prior_grid.GRID with fit_prior(fit=0), is the oracle's total for
  that prior (1e-10 relative, 1e-8 nats) and the same engine's evidence read (1e-12 relative): small_example (both SNP
  orders), tests/example (more than 32 bins per accumulator), a synthetic mixed-type locus, and a locus beyond the
  plain-double range on the register and on the generic kernel.
* The table of a store that is the sum of 2 or 3 rank ranges (pipsort_merge) is the whole pass's.
* The batch equals read_class_evidence on engines created one by one, on 1 and 3 host threads: the same n_configs and empty
  classes, values within 1e-12 relative (separate passes: the kernels' atomic adds land in another order); a bad locus at
  position 17 of 40 stops it with that locus's error, and the next call is right.
* The fit over 30 synthetic loci is at least as good as the best point of a dense evidence grid and lies within a grid step
  of it; the ordinary batch at the fitted prior gives the fit's per-locus totals.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import range_loci as R
from conftest import ROOT, engine_for, oracle_locus, synth_as_oracle_locus, synth_locus
from test_gpu_batch import FAILURES, PIPSORT_E_ARG, PIPSORT_E_SINGULAR, as_dict, bad_locus, expect_error, singular_locus, small_loci
from test_gpu_prior_grid import GRID, with_prior

pytestmark = pytest.mark.gpu


def ntab(c):
    return (c + 1) * (c + 2) // 2


def table_and_evidence(L, c, **kw):
    """One class-resolved engine, one pass: its class table, its evidence read over GRID, U and n_configs."""
    with engine_for(L, c, prior_classes=True, **kw) as e:
        e.reset()
        e.run_exhaustive(c)
        tab = e.read_class_evidence(c)
        ev = e.read_prior_grid(GRID, evidence_only=True)
        return tab, ev[:, 0], e.U, e.config_count()


def evaluate(tab, U, g, p):
    import pipsort_b200 as P
    return P.fit_prior(tab.reshape(1, -1), [U], fit=0, gamma=g, p=p)[2]


def check_table(L, c, oracle_priors=GRID, **kw):
    from oracle import oracle as O
    tab, ev, U, _ = table_and_evidence(L, c, **kw)
    assert tab.shape == (ntab(c),)
    OL = L if hasattr(L, "n_snps") else synth_as_oracle_locus(L)
    for (g, p), want in zip(GRID, ev):
        got = evaluate(tab, U, g, p)
        assert got == pytest.approx(want, rel=1e-12, abs=0), f"gamma={g} p={p}: evidence read"
        if (g, p) in oracle_priors:
            o = O.exhaustive_omp_full(with_prior(OL, g, p), c).total
            assert got == pytest.approx(o, rel=1e-10, abs=1e-8), f"gamma={g} p={p}: oracle"
    return tab


# ---- 1. table against the oracle and the evidence read ----------------------------------------------------------------------
@pytest.mark.parametrize("keep_order", [False, True])
def test_small_example_c3(keep_order):
    tab = check_table(oracle_locus("small_example"), 3, keep_order=keep_order)
    assert np.isfinite(tab[0])


def test_example_c2():
    check_table(oracle_locus("example", p=0.25), 2, oracle_priors=[(0.01, 0.0), (1e-3, 1.0), (0.2, 0.75)])


def test_synthetic_mixed_types():
    check_table(synth_locus(30, overlap=0.5, seed=31), 3)


@pytest.mark.parametrize("generic_only", [False, True])
def test_beyond_the_double_range(generic_only):
    check_table(R.straddle_locus(), 3, oracle_priors=[(0.01, 0.0), (1e-3, 1.0), (0.2, 0.25), (0.01, 0.75)],
                generic_only=generic_only)


def test_empty_classes_are_minus_inf():
    """A locus of 2 union SNPs read at c = 3 has no class with J = 3: -inf, not PostCal's 0.0."""
    from oracle import oracle as O
    one = O.Locus(n_snps=np.array([1, 1], dtype=np.int32), sigma=[np.ones((1, 1)), np.ones((1, 1))],
                  z=[np.array([2.5]), np.array([-1.0])], K=7.25, d=np.array([5.72, 5.72]),
                  snp_map=np.zeros((2, 1), dtype=np.int32), gamma=0.01, p=0.75)
    tab, ev, U, _ = table_and_evidence(one, 3)
    assert np.isfinite(tab[:3]).all()                     # J = 0; J = 1 with a = 0 (one study) and a = 1 (both)
    assert np.isneginf(tab[3:]).all()
    for (g, p), want in zip(GRID, ev):
        assert evaluate(tab, U, g, p) == pytest.approx(want, rel=1e-12)


# ---- 2. sums of stores ------------------------------------------------------------------------------------------------------
def test_merged_stores():
    SL = synth_locus(40, overlap=0.5, seed=99)
    whole, _, U, n = table_and_evidence(SL, 3)
    for parts in (2, 3):
        engines = [engine_for(SL, 3, prior_classes=True) for _ in range(parts)]
        try:
            bounds = engines[0].shard_ranks(3, parts)
            for i, e in enumerate(engines):
                e.reset()
                e.run_exhaustive(3, bounds[i], bounds[i + 1])
            for e in engines[1:]:
                engines[0].merge_from(e)
            tab = engines[0].read_class_evidence(3)
            assert engines[0].config_count() == n
        finally:
            for e in engines:
                e.close()
        assert np.array_equal(np.isneginf(tab), np.isneginf(whole))
        np.testing.assert_allclose(tab, whole, rtol=1e-10, atol=1e-8)
        for g, p in GRID:
            assert evaluate(tab, U, g, p) == pytest.approx(evaluate(whole, U, g, p), rel=1e-10, abs=1e-8)


# ---- 3. batch ---------------------------------------------------------------------------------------------------------------
def one_by_one(D, c):
    import pipsort_b200 as P
    out, cnt = [], []
    for Di in D:
        with P.Engine(Di["num_snps"], Di["sigma"], Di["z"], Di["d"], Di["K"], Di["snp_map"], gamma=Di["gamma"],
                      sharing_param=Di["sharing_param"], max_causal=c, prior_classes=True) as e:
            e.run_exhaustive(c)
            out.append(e.read_class_evidence(c))
            cnt.append(e.config_count())
    return np.array(out), np.array(cnt, dtype=np.uint64)


def table_batch(D, c):
    import pipsort_b200 as P
    B = P.LocusBatch(D, c, class_evidence=True)
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
B = P.LocusBatch(loci, 3, class_evidence=True)
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
    D = [as_dict(L) for L in small_loci()]
    want, wcnt = one_by_one(D, 3)
    same_tables(*table_batch(D, 3), want, wcnt)              # three host threads
    src, dst = tmp_path / "loci.npz", tmp_path / "tables.npz"
    np.savez(src, n=len(D), **{f"{k}{i}": v for i, L in enumerate(D) for k, v in L.items()})
    env = dict(os.environ, PIPSORT_BATCH_THREADS="1")
    p = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(src), str(dst)], capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    out = np.load(dst)
    same_tables(out["tab"], out["cnt"], want, wcnt)


@pytest.mark.parametrize("kind", list(FAILURES))
def test_failure_inside_a_batch(kind):
    D = [as_dict(L) for L in small_loci()]
    want, wcnt = table_batch(D, 3)
    code, text = FAILURES[kind]
    bad = list(D)
    bad[17] = bad_locus(kind)
    expect_error(code, text, table_batch, bad, 3)
    same_tables(*table_batch(D, 3), want, wcnt)


# ---- 4. the fit ---------------------------------------------------------------------------------------------------------------
def fit_loci():
    """30 loci: strong SNPs shared by both studies in some, present in one study only in others (overlap 0 .. 1)."""
    from pipsort_b200 import synth
    return [as_dict(synth.make_locus(10 + (i % 5) * 4, overlap=(0.0, 0.3, 0.6, 1.0, 0.9)[i % 5], seed=900 + i)) for i in range(30)]


def test_fit_against_evidence_grids():
    import pipsort_b200 as P
    D = fit_loci()
    U = [L["snp_map"].shape[1] for L in D]
    tabs = P.class_evidence_batch(D, 3)
    # p alone, gamma = 0.01: a 1e-3-spaced grid over (0, 1]
    ps = np.round(np.arange(1, 1001) * 1e-3, 12)
    ev = P.posterior_exhaustive_grid_batch(D, 3, [(0.01, float(p)) for p in ps], evidence_only=True)[:, :, 0].sum(0)
    g, p, joint, per = P.fit_prior(tabs, U, fit="p", gamma=0.01)
    k = int(np.argmax(ev))
    assert g == 0.01
    assert joint >= ev[k] - 1e-9
    assert abs(p - ps[k]) <= 1e-3 + 1e-12
    # (gamma, p) against a 2-D grid: log-spaced gamma x p
    gs = np.geomspace(1e-4, 0.3, 40)
    ps2 = np.round(np.arange(1, 51) * 0.02, 12)
    pri = [(float(a), float(b)) for a in gs for b in ps2]
    ev2 = P.posterior_exhaustive_grid_batch(D, 3, pri, evidence_only=True)[:, :, 0].sum(0).reshape(len(gs), len(ps2))
    g2, p2, joint2, per2 = P.fit_prior(tabs, U, fit="gamma,p")
    i, j = np.unravel_index(int(np.argmax(ev2)), ev2.shape)
    assert joint2 >= ev2[i, j] - 1e-9
    step = np.log(gs[1] / gs[0])
    assert abs(np.log(g2) - np.log(gs[i])) <= step * (1 + 1e-9)
    assert abs(p2 - ps2[j]) <= 0.02 + 1e-12
    # the PIPs at the fitted prior: the ordinary batch, whose totals are the fit's per-locus values
    for gg, pp, want in ((g, p, per), (g2, p2, per2)):
        res = P.posterior_exhaustive_batch([dict(L, gamma=gg, sharing_param=pp) for L in D], 3)
        np.testing.assert_allclose([r.total for r in res], want, rtol=1e-10, atol=0)


# ---- 5. refusals --------------------------------------------------------------------------------------------------------------
def test_refusals():
    SL = synth_locus(20, overlap=0.5, seed=3)
    with engine_for(SL, 3) as e:
        e.compute_total_likelihood(3)
        expect_error(PIPSORT_E_ARG, "PIPSORT_PRIOR_CLASSES", e.read_class_evidence, 3)
    with engine_for(SL, 3, prior_classes=True) as e:
        e.run_exhaustive(3)
        expect_error(PIPSORT_E_ARG, "c=4", e.read_class_evidence, 4)
        expect_error(PIPSORT_E_ARG, "c=-1", e.read_class_evidence, -1)
        assert np.isfinite(e.read_class_evidence(3)[0])
    with engine_for(singular_locus()[0], 3, prior_classes=True) as e:
        e.run_exhaustive(3)
        expect_error(PIPSORT_E_SINGULAR, "matrix is singular", e.read_class_evidence, 3)
