"""A grid of priors for a list of loci in one call (pipsort_posterior_exhaustive_grid_batch, LocusBatch with priors) and the
evidence read (total and noCausal only, every per-SNP member of the output blocks NULL).

Every (locus, prior) result must be what an ordinary engine created with that prior reports for that locus: the one-call
posterior_exhaustive with that prior (same n_configs, 1e-12 relative, the same empty pattern at p = 1), the one-call grid,
the ordinary batch at one prior, and the oracle on a subset.  The loci are those of test_gpu_batch.py (40 distinct small
loci, the range loci at c = 1 .. 5, degenerate loci, tests/example, raw LD); the grids those of test_gpu_prior_grid.py.

Before every run() the result buffer is filled with NaN and the counts with 0, so that an output slot that is never written
cannot keep a right answer from an earlier call.
"""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_results_match, engine_for, oracle_locus, synth_locus
from test_gpu_batch import (FAILURES, HARD, PIPSORT_E_ARG, RTOL_SAME, as_dict, as_oracle, assert_each, bad_locus, batch,  # noqa: F401
                            edge_loci, expect_error, golden_locus, one_call, pool_used, same, small_loci)
from test_gpu_extended_range import locus as range_locus
from test_gpu_extended_range import synth12
from test_gpu_prior_grid import GRID, SMALL_GRID, match_oracle, with_prior

pytestmark = pytest.mark.gpu

PER_SNP = ("postValues", "sharedPips", "sharedLL", "notSharedLL")


def run_fresh(B):
    """B.run() into a result buffer of NaN and counts of 0; the results (evidence() for an evidence batch), copied out."""
    B.buf.fill(np.nan)
    B.cnt[:] = 0
    B.run()
    return copy.deepcopy(B.evidence() if B.evidence_only else B.results())


def grid_batch(D, c, priors, raw_ld=False, evidence_only=False):
    import pipsort_b200 as P
    return run_fresh(P.LocusBatch(D, c, raw_ld=raw_ld, priors=priors, evidence_only=evidence_only))


def one_call_grid(D, c, priors, raw_ld=False):
    import pipsort_b200 as P
    return P.posterior_exhaustive_grid(D["num_snps"], D["sigma"], D["z"], D["d"], D["K"], D["snp_map"], c, priors, raw_ld=raw_ld)


def scalars(r):
    return np.array([r.total, r.noCausal[0], r.noCausal[1]])


def each_pair(got, priors, cmp):
    """cmp(got[i][j], i, j, gamma, p) for every locus i and prior j; a failure names both."""
    for i, row in enumerate(got):
        assert len(row) == len(priors)
        for j, (g, p) in enumerate(priors):
            try:
                cmp(row[j], i, j, g, p)
            except AssertionError as err:
                raise AssertionError(f"locus {i}, prior {j} (gamma={g}, p={p}): {err}") from None


def vs_ordinary(got, D, c, priors):
    """Every (locus, prior) against posterior_exhaustive with that prior and against the one-call grid of the locus."""
    grids = [one_call_grid(Di, c, priors) for Di in D]

    def cmp(r, i, j, g, p):
        same(r, one_call(dict(D[i], gamma=g, sharing_param=p), c))
        same(r, grids[i][j])
    each_pair(got, priors, cmp)


def same_evidence(ev, full):
    """ev [n_loci, n_priors, 3] against the scalars of full results, 1e-12 relative and the same zeros."""
    want = np.array([[scalars(r) for r in row] for row in full])
    assert ev.shape == want.shape
    assert np.array_equal(ev == 0, want == 0)
    np.testing.assert_allclose(ev, want, rtol=RTOL_SAME, atol=0)


# ---- 1. 40 distinct loci x the wide grid ------------------------------------------------------------------------------------
def test_distinct_loci_wide_grid():
    """40 small loci x 18 priors (p = 0, 1e-9, 0.25, 0.75, 0.999999, 1; gamma = 1e-3, 0.01, 0.2) on three threads: each pair
    against the ordinary one-call path with that prior and the one-call grid, a subset against the oracle; the evidence batch
    against the full one."""
    from oracle import oracle as O
    loci = small_loci()
    D = [as_dict(L) for L in loci]
    got = grid_batch(D, 3, GRID)
    vs_ordinary(got, D, 3, GRID)
    for i in (0, 17, 39):
        for j in (0, 5, 7, 16):
            g, p = GRID[j]
            match_oracle(got[i][j], O.exhaustive_omp_full(with_prior(as_oracle(loci[i]), g, p), 3))
    same_evidence(grid_batch(D, 3, GRID, evidence_only=True), got)


@pytest.mark.parametrize("prior", [(0.01, 0.75), (1e-3, 1.0), (0.2, 0.0)])
def test_one_prior_equals_ordinary_batch(prior):
    D = [as_dict(L, gamma=prior[0], sharing_param=prior[1]) for L in small_loci()]
    want = batch(D, 3)
    got = grid_batch(D, 3, [prior])
    assert_each([row[0] for row in got], want, same)


# ---- 2. the kernels' paths, degenerate loci, tests/example, raw LD ----------------------------------------------------------
@pytest.mark.parametrize("c", [1, 2, 3, 4, 5])
def test_range_loci(c):
    """Loci that leave the fast range (fast and slow paths of the register kernel; the generic kernel for the classes above
    3 at c = 4, 5) next to a small synthetic locus."""
    names = HARD if c == 3 else ("straddle",)
    D = [as_dict(range_locus(n)) for n in names] + [as_dict(synth12())]
    vs_ordinary(grid_batch(D, c, SMALL_GRID), D, c, SMALL_GRID)


def test_edge_loci_and_example_in_a_batch():
    """No SNP at all, a study without SNPs, c > U, and tests/example (more than 32 bins per accumulator) at c = 2 among
    ordinary loci; the example's own prior against its golden dump."""
    g, prm, EX = golden_locus("example_c2_p025")
    priors = SMALL_GRID + [(prm["gamma"], prm["p"])]
    D = [as_dict(L) for L in small_loci()[:6]]
    for pos, L in zip((1, 4, 5, 8), edge_loci()[:2] + [EX] + edge_loci()[2:]):
        D.insert(pos, as_dict(L))
    got = grid_batch(D, 2, priors)
    vs_ordinary(got, D, 2, priors)
    assert got[5][-1].n_configs == 216817
    assert_results_match(got[5][-1], g)
    same_evidence(grid_batch(D, 2, priors, evidence_only=True), got)


def test_raw_ld_grid_batch():
    """Nine loci from the raw small_example files (PIPSORT_RAW_LD), the d settings of three golden dumps interleaved, the
    priors of the three dumps: each locus's own prior against its dump, every prior against the one-call grid."""
    from oracle import oracle as O
    from conftest import dataset_paths
    ld_files, z_files, _, _ = dataset_paths("small_example")
    lds, zs = [O.read_ld(f) for f in ld_files], [O.read_z(f)[1] for f in z_files]
    names = ("small_c3_p075", "small_c3_p0", "small_c3_g005_t1_s3")
    gl = [golden_locus(n) for n in names]
    priors = [(L.gamma, L.p) for _, _, L in gl]
    D, want = [], []
    for k in range(9):
        g, prm, L = gl[k % 3]
        D.append(dict(num_snps=L.n_snps, sigma=np.concatenate([ld.ravel() for ld in lds]), z=np.concatenate(zs), d=L.d, K=0.0,
                      snp_map=L.snp_map, gamma=L.gamma, sharing_param=L.p))
        want.append(g)
    got = grid_batch(D, 3, priors, raw_ld=True)
    for k, row in enumerate(got):
        assert row[k % 3].n_configs == 268, f"locus {k}"
        assert_results_match(row[k % 3], want[k])
        for r, w in zip(row, one_call_grid(D[k], 3, priors, raw_ld=True)):
            same(r, w)


# ---- 3. the evidence read ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["synth150", "example"])
def test_evidence_read_is_bit_identical(which):
    """On one engine, read_prior_grid(evidence_only=True) gives the scalars of the full read bit for bit (the same store;
    the example locus has more than 32 bins per accumulator)."""
    L, c = (synth_locus(150), 3) if which == "synth150" else (oracle_locus("example", p=0.25), 2)
    with engine_for(L, c, prior_classes=True) as e:
        e.reset()
        e.run_exhaustive(c)
        full = e.read_prior_grid(GRID)
        ev = e.read_prior_grid(GRID, evidence_only=True)
        again = e.read_prior_grid(GRID)
    assert ev.shape == (len(GRID), 3)
    want = np.array([scalars(r) for r in full])
    assert np.array_equal(ev, want)
    assert np.array_equal(np.array([scalars(r) for r in again]), want)


def test_null_members_are_never_written():
    """Locus 3's blocks leave every per-SNP member NULL (an evidence read among full ones); locus 6's block for prior 2
    leaves postValues and sharedLL NULL (a full read).  What those members would point to stays NaN; everything else is
    what the full grid batch gives."""
    import pipsort_b200 as P
    D = [as_dict(L) for L in small_loci()[:10]]
    k = len(SMALL_GRID)
    full = grid_batch(D, 3, SMALL_GRID)
    B = P.LocusBatch(D, 3, priors=SMALL_GRID)
    for j in range(k):
        for m in PER_SNP:
            B.oa[3 * k + j][m] = 0
    for m in ("postValues", "sharedLL"):
        B.oa[6 * k + 2][m] = 0
    got = run_fresh(B)
    for i in range(len(D)):
        for j in range(k):
            g, w = got[i][j], full[i][j]
            if i == 3 or (i, j) == (6, 2):
                nulls = PER_SNP if i == 3 else ("postValues", "sharedLL")
                for m in PER_SNP:
                    a, b = getattr(g, m), getattr(w, m)
                    if m in nulls:
                        assert np.isnan(a).all(), f"locus {i}, prior {j}: {m} was written"
                    else:
                        np.testing.assert_allclose(a, b, rtol=RTOL_SAME, atol=0)
                np.testing.assert_allclose(scalars(g), scalars(w), rtol=RTOL_SAME, atol=0)
                assert g.n_configs == w.n_configs
            else:
                same(g, w)


# ---- 4. host threads --------------------------------------------------------------------------------------------------------
def test_seven_and_eight_loci_agree():
    """7 loci run on one host thread, 8 on three: the 7 leading loci come back the same either way, full and evidence."""
    D = [as_dict(L) for L in small_loci()[:8]]
    seven, eight = grid_batch(D[:7], 3, SMALL_GRID), grid_batch(D, 3, SMALL_GRID)
    each_pair(eight[:7], SMALL_GRID, lambda r, i, j, g, p: same(r, seven[i][j]))
    same_evidence(grid_batch(D[:7], 3, SMALL_GRID, evidence_only=True), seven)
    same_evidence(grid_batch(D, 3, SMALL_GRID, evidence_only=True), eight)


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
B = P.LocusBatch(loci, int(src["c"]), priors=src["priors"].tolist())
B.buf.fill(np.nan)
B.cnt[:] = 0
B.run()
np.savez(sys.argv[3], buf=B.buf, cnt=B.cnt)
"""


@pytest.mark.parametrize("threads", [1, 2, 8])
def test_other_thread_counts(threads, tmp_path):
    """The 40-locus grid batch with PIPSORT_BATCH_THREADS = 1, 2 and 8 (read once per process: in a child process) gives
    what the default three threads give in this process."""
    import pipsort_b200 as P
    D = [as_dict(L) for L in small_loci()]
    src, dst = tmp_path / "loci.npz", tmp_path / "results.npz"
    np.savez(src, n=len(D), c=3, priors=np.array(SMALL_GRID), **{f"{k}{i}": v for i, L in enumerate(D) for k, v in L.items()})
    env = dict(os.environ, PIPSORT_BATCH_THREADS=str(threads))
    p = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(src), str(dst)], capture_output=True, text=True, env=env,
                       timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    B = P.LocusBatch(D, 3, priors=SMALL_GRID)
    want = run_fresh(B)
    out = np.load(dst)
    B.buf[:] = out["buf"]                                       # the same layout: slice the child's buffer as this one
    B.cnt[:] = out["cnt"]
    each_pair(B.results(), SMALL_GRID, lambda r, i, j, g, p: same(r, want[i][j]))


# ---- 5. failures ------------------------------------------------------------------------------------------------------------
def test_bad_prior_fails_before_any_engine(pool_used):
    """A bad prior is reported even though locus 0 would be refused at create: no engine was made; the pool is untouched."""
    import pipsort_b200 as P
    D = [as_dict(L) for L in small_loci()]
    D[0] = bad_locus("d")
    base = pool_used()
    for bad, what in (((0.01, 1.5), "sharing_param"), ((1.0, 0.5), "gamma"), ((float("nan"), 0.5), "gamma")):
        for ev in (False, True):
            err = expect_error(PIPSORT_E_ARG, "prior 1", run_fresh, P.LocusBatch(D, 3, priors=[(0.01, 0.75), bad], evidence_only=ev))
            assert what in str(err) and "d[1]" not in str(err)
    assert pool_used() == base


@pytest.mark.parametrize("kind", list(FAILURES))
def test_failure_inside_a_grid_batch(kind, pool_used):
    """One bad locus at position 17 of 40 (worker thread 2 of 3): the call returns its error on the calling thread, every
    engine still in flight is destroyed, and the next grid batch in the process is right."""
    import pipsort_b200 as P
    code, text = FAILURES[kind]
    good = P.LocusBatch([as_dict(L) for L in small_loci()], 3, priors=SMALL_GRID)
    want = run_fresh(good)              # warm-up: the streams, events and pinned staging of the engines in flight
    base = pool_used()
    D = [as_dict(L) for L in small_loci()]
    D[17] = bad_locus(kind)
    for ev in (False, True):
        expect_error(code, text, run_fresh, P.LocusBatch(D, 3, priors=SMALL_GRID, evidence_only=ev))
        assert text in P.lib().pipsort_last_error().decode()
        assert pool_used() == base
    each_pair(run_fresh(good), SMALL_GRID, lambda r, i, j, g, p: same(r, want[i][j]))
    vs_ordinary([want[i] for i in (16, 17, 18)], [as_dict(small_loci()[i]) for i in (16, 17, 18)], 3, SMALL_GRID)
