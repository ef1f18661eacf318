"""The calls a user with many loci makes -- pipsort_posterior_exhaustive_batch and the one-call pipsort_posterior_exhaustive --
against the oracle, the golden dumps and the step-by-step Engine path.

* Distinct loci on several host threads: 40 small synthetic loci (every thread reuses its three pipeline slots several
  times), 24 headline-size loci read from pinned host memory with one U and four type layouts, the switch from one thread
  to three at 8 loci, and 1 / 2 / 8 threads in child processes (PIPSORT_BATCH_THREADS is read once per process).
* The pair tables these calls build in pipsort_create's own preparation launch: on loci that leave the fast range (c = 1
  .. 5), on degenerate loci (no SNP at all, a study without SNPs, c > U), on tests/example (more than 32 bins per
  accumulator: the scanning finalize), and on raw LD (PIPSORT_RAW_LD) from three threads at once.
* Failures inside a batch -- refused at create, a refused argument, a singular block found by the kernel and reported when
  the locus is read: the error reaches the calling thread, every engine goes back to the pool, the next batch is right.
* A locus with an indefinite 2x2 block: every path that evaluates the block reports PIPSORT_E_SINGULAR; work that avoids
  it matches the oracle.

Before every run() the result buffer is filled with NaN and the counts with 0, so that an output slot that is never written
cannot keep a right answer from an earlier call.  Against the Engine path the tolerance is 1e-12 relative: the kernels are
the same, only the order of the atomics differs.
"""
import copy
import ctypes as C
import dataclasses
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, args_to_params, assert_results_match, dataset_paths, engine_for, golden, oracle_locus, synth_as_oracle_locus
from test_gpu_extended_range import check, oracle_exh
from test_gpu_extended_range import locus as range_locus
from test_gpu_extended_range import n_configs as range_n_configs

pytestmark = pytest.mark.gpu

PIPSORT_E_ARG, PIPSORT_E_RANGE, PIPSORT_E_SINGULAR = 1, 4, 5
RTOL_SAME = 1e-12
CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7


@pytest.fixture(scope="module")
def pool_used():
    """() -> bytes of device 0's default memory pool in use, once all work on the device has completed."""
    cu = C.CDLL("libcuda.so.1")
    dev, ctx, pool = C.c_int(), C.c_void_p(), C.c_void_p()
    assert cu.cuInit(0) == 0
    assert cu.cuDeviceGet(C.byref(dev), 0) == 0
    assert cu.cuDevicePrimaryCtxRetain(C.byref(ctx), dev) == 0      # the context the engine's runtime calls use
    assert cu.cuCtxSetCurrent(ctx) == 0
    assert cu.cuDeviceGetDefaultMemPool(C.byref(pool), dev) == 0

    def used():
        assert cu.cuCtxSynchronize() == 0
        v = C.c_uint64()
        assert cu.cuMemPoolGetAttribute(pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, C.byref(v)) == 0
        return v.value
    yield used
    cu.cuDevicePrimaryCtxRelease(dev)


# ---- helpers --------------------------------------------------------------------------------------------------------------
def as_dict(L, **over):
    """A SynthLocus or oracle Locus as the dict posterior_exhaustive's arguments / LocusBatch take (flat sigma and z)."""
    n = L.num_snps if hasattr(L, "num_snps") else L.n_snps
    p = L.sharing_param if hasattr(L, "sharing_param") else L.p
    D = dict(num_snps=np.asarray(n, dtype=np.int32), sigma=np.concatenate([np.asarray(s, dtype=np.float64).ravel() for s in L.sigma]),
             z=np.concatenate([np.asarray(v, dtype=np.float64).ravel() for v in L.z]), d=np.asarray(L.d, dtype=np.float64),
             K=float(L.K), snp_map=np.asarray(L.snp_map, dtype=np.int32), gamma=float(L.gamma), sharing_param=float(p))
    D.update(over)
    return D


def as_oracle(L):
    return L if hasattr(L, "n_snps") else synth_as_oracle_locus(L)


def one_call(D, c):
    import pipsort_b200 as P
    return P.posterior_exhaustive(D["num_snps"], D["sigma"], D["z"], D["d"], D["K"], D["snp_map"], c, gamma=D["gamma"],
                                  sharing_param=D["sharing_param"])


def run_fresh(B):
    """B.run() into a result buffer of NaN and counts of 0; the per-locus results, copied out of the buffer."""
    B.buf.fill(np.nan)
    B.cnt[:] = 0
    B.run()
    return copy.deepcopy(B.results())


def batch(loci, c, raw_ld=False):
    import pipsort_b200 as P
    return run_fresh(P.LocusBatch(loci, c, raw_ld=raw_ld))


def vs_oracle(got, want):
    assert got.n_configs == want.n_eval
    assert_results_match(got, want)


def same(got, want):
    assert got.n_configs == want.n_configs
    assert_results_match(got, want, rtol=RTOL_SAME)


def assert_each(got, want, cmp):
    """cmp(got[i], want[i]) for every locus; a failure names the locus."""
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        try:
            cmp(g, w)
        except AssertionError as err:
            raise AssertionError(f"locus {i}: {err}") from None


def expect_error(code, text, f, *a, **kw):
    import pipsort_b200 as P
    with pytest.raises(P.PipsortError) as ei:
        f(*a, **kw)
    assert ei.value.code == code, str(ei.value)
    assert text in str(ei.value)
    return ei.value


# ---- loci, once per session ------------------------------------------------------------------------------------------------
OVERLAPS = (0.0, 0.5, 0.8, 1.0)
GAMMAS = (1e-3, 0.01, 0.2)
SHARING = (0.0, 1e-9, 0.25, 0.75, 0.999999)


@functools.lru_cache(maxsize=None)
def small_loci():
    """40 distinct loci for c = 3: 12 .. 60 SNPs per study, the overlaps, gammas and sharing parameters above in turn."""
    from pipsort_b200 import synth
    return [synth.make_locus(12 + 48 * i // 39, overlap=OVERLAPS[i % 4], seed=600 + i, gamma=GAMMAS[i % 3],
                             sharing_param=SHARING[i % 5]) for i in range(40)]


@functools.lru_cache(maxsize=None)
def small_oracle(c=3):
    from oracle import oracle as O
    return [O.exhaustive_omp_full(as_oracle(L), c) for L in small_loci()]


# (SNPs per study, overlap): U = 180 each, four different type layouts (the exhaustive work plan is cached per U and layout)
LAYOUTS = ((150, 0.8), (144, 0.75), (120, 0.5), (90, 0.0))


@functools.lru_cache(maxsize=None)
def headline_loci():
    """24 loci, the four layouts in turn, six seeds each."""
    from pipsort_b200 import synth
    return [synth.make_locus(n, overlap=ov, seed=900 + 10 * j + k) for j in range(6) for k, (n, ov) in enumerate(LAYOUTS)]


@functools.lru_cache(maxsize=None)
def singular_locus():
    """make_locus(12, overlap=0.5) with Sigma_0[i][j] = Sigma_0[j][i] = 1.5 for two shared SNPs i, j: then
    det(I + d Sigma_{i,j}) = (1 + d)^2 - (1.5 d)^2 < 0 for d > 2 (study 0's d is 26.5), and the Schur complement of the
    pair is about -30 in either order, far from the kernels' guard at 0.25.  Returns (locus, the pair as union positions,
    the pair as study-0 indices)."""
    from pipsort_b200 import synth
    SL = synth.make_locus(12, overlap=0.5, seed=41)
    smap = SL.snp_map
    shared = np.nonzero((smap[0] >= 0) & (smap[1] >= 0))[0]
    g = (int(shared[1]), int(shared[3]))
    i, j = int(smap[0, g[0]]), int(smap[0, g[1]])
    sig0 = np.array(SL.sigma[0])
    sig0[i, j] = sig0[j, i] = 1.5
    L = dataclasses.replace(SL, sigma=[sig0, SL.sigma[1]])
    d = float(L.d[0])
    schur = 1.0 + d * sig0[j, j] - (d * 1.5) ** 2 / (1.0 + d * sig0[i, i])
    assert d > 20 and schur < -20
    return L, g, (i, j)


# ---- 1. distinct loci on several host threads -------------------------------------------------------------------------------
def test_distinct_small_loci_on_three_threads():
    """40 loci >= 3 threads x 3 pipeline slots + 1: every thread reuses its slots; three calls on one LocusBatch, as the
    benchmark makes them, each against the oracle."""
    import pipsort_b200 as P
    B = P.LocusBatch([as_dict(L) for L in small_loci()], 3)
    for _ in range(3):
        assert_each(run_fresh(B), small_oracle(), vs_oracle)


def test_headline_size_loci_from_pinned_memory():
    """24 distinct 150-SNP-class loci (U = 180, four type layouts) whose sigma and z are pinned host memory, as the benchmark
    builds them: the uploads of pipsort_create are then truly asynchronous.  Every locus against the Engine path, two of
    them against the oracle."""
    import torch
    import pipsort_b200 as P
    from oracle import oracle as O
    loci = headline_loci()
    assert {L.U for L in loci} == {180} and len({L.n_types() for L in loci}) == len(LAYOUTS)
    keep, D = [], []
    for L in loci:
        sg = torch.from_numpy(np.concatenate([s.ravel() for s in L.sigma])).pin_memory()
        zz = torch.from_numpy(np.concatenate(L.z)).pin_memory()
        assert sg.is_pinned() and zz.is_pinned()
        keep += [sg, zz]
        D.append(as_dict(L, sigma=sg.numpy(), z=zz.numpy()))
    B = P.LocusBatch(D, 3)
    assert all(B.la["sigma"][i] == D[i]["sigma"].ctypes.data for i in range(len(D)))     # the batch reads the pinned arrays
    want = []
    for L in loci:
        with engine_for(L, 3) as e:
            want.append(e.compute_total_likelihood(3))
    assert len({w.total for w in want}) == len(loci)            # equal shapes, different data: no two results alike
    for _ in range(2):
        got = run_fresh(B)
        assert_each(got, want, same)
    for i in (0, 2):                                            # layouts (150, 0.8) and (120, 0.5)
        vs_oracle(got[i], O.exhaustive_omp_full(as_oracle(loci[i]), 3))


def test_seven_and_eight_loci_agree():
    """7 loci run on one host thread, 8 on three: the 7 leading loci come back the same either way."""
    D = [as_dict(L) for L in small_loci()[:8]]
    seven = batch(D[:7], 3)
    eight = batch(D, 3)
    assert_each(eight[:7], seven, same)
    assert_each(eight, small_oracle()[:8], vs_oracle)


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
B = P.LocusBatch(loci, int(src["c"]))
B.buf.fill(np.nan)
B.cnt[:] = 0
B.run()
np.savez(sys.argv[3], buf=B.buf, cnt=B.cnt)
"""


@pytest.mark.parametrize("threads", [1, 2, 8])
def test_other_thread_counts(threads, tmp_path):
    """The 40-locus batch with PIPSORT_BATCH_THREADS = 1, 2 and 8 (read once per process: in a child process) gives what
    the default three threads give in this process."""
    import pipsort_b200 as P
    D = [as_dict(L) for L in small_loci()]
    src, dst = tmp_path / "loci.npz", tmp_path / "results.npz"
    np.savez(src, n=len(D), c=3, **{f"{k}{i}": v for i, L in enumerate(D) for k, v in L.items()})
    env = dict(os.environ, PIPSORT_BATCH_THREADS=str(threads))
    p = subprocess.run([sys.executable, "-c", CHILD, ROOT, str(src), str(dst)], capture_output=True, text=True, env=env,
                       timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    B = P.LocusBatch(D, 3)
    want = run_fresh(B)
    out = np.load(dst)
    B.buf[:] = out["buf"]                                       # the same layout: slice the child's buffer as this one
    B.cnt[:] = out["cnt"]
    assert_each(B.results(), want, same)


# ---- 2. pair tables built in the creation launch ---------------------------------------------------------------------------
HARD = ("straddle", "threshold", "lone", "spread")


@pytest.mark.parametrize("name", HARD)
def test_hard_loci_one_call(name):
    """Loci that leave the fast range (range_loci.py): the pair table's +inf entries send subsets down the mantissa/exponent
    path; here the tables come from pipsort_create's own launch, not from the Engine path's lazy builder."""
    check(one_call(as_dict(range_locus(name)), 3), oracle_exh(name, 3), range_n_configs(name, 3))


@pytest.mark.parametrize("c", [1, 2, 4, 5])
def test_straddle_one_call_other_classes(c):
    """c = 1 builds no table, c = 2 the tables of the pairs only, c = 4 / 5 run the generic kernel for the classes above 3
    next to the register kernel with the fused tables."""
    check(one_call(as_dict(range_locus("straddle")), c), oracle_exh("straddle", c), range_n_configs("straddle", c))


def test_hard_loci_batch():
    names = HARD + HARD
    got = batch([as_dict(range_locus(n)) for n in names], 3)
    for i, (name, r) in enumerate(zip(names, got)):
        try:
            check(r, oracle_exh(name, 3), range_n_configs(name, 3))
        except AssertionError as err:
            raise AssertionError(f"locus {i} ({name}): {err}") from None


def edge_loci():
    """The loci of test_gpu_parity's test_edge_cases_empty_and_ragged: no SNP at all, study 1 without SNPs (its table is
    the zero row alone), one shared SNP with c = 3 > U."""
    from oracle import oracle as O
    from pipsort_b200 import synth
    empty = O.Locus(n_snps=np.array([0, 0], dtype=np.int32), sigma=[np.zeros((0, 0)), np.zeros((0, 0))], z=[np.zeros(0), np.zeros(0)],
                    K=3.0, d=np.array([5.72, 5.72]), snp_map=np.zeros((2, 0), dtype=np.int32), gamma=0.01, p=0.75)
    SL = synth.make_locus(4, overlap=0.0, seed=9)
    ragged = O.Locus(n_snps=np.array([4, 0], dtype=np.int32), sigma=[SL.sigma[0], np.zeros((0, 0))], z=[SL.z[0], np.zeros(0)],
                     K=1.25, d=SL.d, snp_map=np.array([[0, 1, 2, 3], [-1, -1, -1, -1]], dtype=np.int32), gamma=0.01, p=0.75)
    one = O.Locus(n_snps=np.array([1, 1], dtype=np.int32), sigma=[np.ones((1, 1)), np.ones((1, 1))], z=[np.array([2.5]), np.array([-1.0])],
                  K=7.25, d=np.array([5.72, 5.72]), snp_map=np.zeros((2, 1), dtype=np.int32), gamma=0.01, p=0.75)
    return [empty, ragged, one]


def test_edge_loci_one_call_and_batch():
    from oracle import oracle as O
    E = edge_loci()
    want = [O.exhaustive(L, 3) for L in E]
    assert [w.n_eval for w in want] == [1, 1 + 4 + 6 + 4, 4]
    assert want[0].total == pytest.approx(-3.0 / 2 - 1.0, rel=1e-14)
    assert_each([one_call(as_dict(L), 3) for L in E], want, vs_oracle)
    # each next to ordinary loci in a batch of 9 (three threads): positions 1, 4 and 8
    D = [as_dict(L) for L in small_loci()[:6]]
    W = list(small_oracle()[:6])
    for pos, L, w in zip((1, 4, 8), E, want):
        D.insert(pos, as_dict(L))
        W.insert(pos, w)
    assert_each(batch(D, 3), W, vs_oracle)


def golden_locus(name):
    g = golden(name)
    prm = args_to_params(g["args"])
    return g, prm, oracle_locus(g["dataset"], p=prm["p"], gamma=prm["gamma"], s=prm["s"], t=prm["t"])


def test_c2_batch_matches_golden_dumps():
    """tests/example (~80 bins per accumulator: the scanning finalize, inside the pipeline) and small_example at c = 2 in
    one batch with synthetic loci, each against its golden dump / the oracle."""
    gl = [golden_locus(n) for n in ("example_c2_p025", "small_c2_p025", "small_c2_p075")]
    assert all(prm["c"] == 2 for _, prm, _ in gl)
    pad = small_loci()[:6]
    D = [as_dict(L) for L in pad[:4]] + [as_dict(L) for _, _, L in gl] + [as_dict(L) for L in pad[4:]]
    got = batch(D, 2)
    for r, (g, _, _), n in zip(got[4:7], gl, (216817, 76, 76)):
        assert r.n_configs == n
        assert_results_match(r, g)
    assert_each(got[:4] + got[7:], small_oracle(2)[:6], vs_oracle)


def test_raw_ld_batch_matches_golden_dumps():
    """Nine loci from the raw small_example files (PIPSORT_RAW_LD: PSD shift, eigen-decomposition, fused tables on the
    device), the prior / d settings of three golden dumps interleaved: three threads pre-process at once."""
    from oracle import oracle as O
    ld_files, z_files, _, _ = dataset_paths("small_example")
    lds, zs = [O.read_ld(f) for f in ld_files], [O.read_z(f)[1] for f in z_files]
    D, want = [], []
    for k in range(9):
        g, prm, L = golden_locus(("small_c3_p075", "small_c3_p0", "small_c3_g005_t1_s3")[k % 3])
        assert prm["c"] == 3
        D.append(dict(num_snps=L.n_snps, sigma=np.concatenate([ld.ravel() for ld in lds]), z=np.concatenate(zs), d=L.d, K=0.0,
                      snp_map=L.snp_map, gamma=L.gamma, sharing_param=L.p))
        want.append(g)
    got = batch(D, 3, raw_ld=True)
    for i, (r, g) in enumerate(zip(got, want)):
        assert r.n_configs == 268, f"locus {i}"
        assert_results_match(r, g)


# ---- 4. failures inside a batch ---------------------------------------------------------------------------------------------
def bad_locus(kind):
    base = small_loci()[17]
    if kind == "range":                 # as test_out_of_range_locus_is_refused: refused at create
        D = as_dict(base)
        D["z"][0] = 1e6
        return D
    if kind == "d":
        return as_dict(base, d=np.array([float(base.d[0]), 0.0]))
    return as_dict(singular_locus()[0])     # found by the exhaustive kernel, reported when the locus is read


FAILURES = {"range": (PIPSORT_E_RANGE, "exponent range"), "d": (PIPSORT_E_ARG, "d[1]"),
            "singular": (PIPSORT_E_SINGULAR, "matrix is singular")}


@pytest.mark.parametrize("kind", list(FAILURES))
def test_failure_inside_a_batch(kind, pool_used):
    """One bad locus at position 17 of 40 (worker thread 2 of 3): the call returns its error on the calling thread, every
    engine still in flight is destroyed, and the next batch in the process is right."""
    import pipsort_b200 as P
    code, text = FAILURES[kind]
    good = P.LocusBatch([as_dict(L) for L in small_loci()], 3)
    run_fresh(good)                     # warm-up: the streams, events and pinned staging of the engines in flight
    base = pool_used()
    D = [as_dict(L) for L in small_loci()]
    D[17] = bad_locus(kind)
    expect_error(code, text, run_fresh, P.LocusBatch(D, 3))
    assert text in P.lib().pipsort_last_error().decode()
    assert pool_used() == base
    assert_each(run_fresh(good), small_oracle(), vs_oracle)


# ---- 5. a singular block on every path --------------------------------------------------------------------------------------
@pytest.mark.parametrize("c,generic_only", [(2, False), (3, False), (3, True), (4, False)])
def test_singular_block_exhaustive(c, generic_only):
    L = singular_locus()[0]
    with engine_for(L, c, generic_only=generic_only) as e:
        expect_error(PIPSORT_E_SINGULAR, "matrix is singular", e.compute_total_likelihood, c)


@pytest.mark.parametrize("c", [2, 3])
def test_singular_block_one_call(c):
    expect_error(PIPSORT_E_SINGULAR, "matrix is singular", one_call, as_dict(singular_locus()[0]), c)


def test_singular_locus_class_1():
    """Size class 1 never forms the pair: the engine and the one-call path match the oracle."""
    from oracle import oracle as O
    L = singular_locus()[0]
    want = O.exhaustive(as_oracle(L), 1)
    with engine_for(L, 3) as e:
        vs_oracle(e.compute_total_likelihood(1), want)
    vs_oracle(one_call(as_dict(L), 1), want)


def union_rows(rng, n, kmax, with_pair):
    """n rows of union positions (snp_map order, -1 padded): every row holds both SNPs of the singular pair, or none holds
    both (but many hold one of them)."""
    L, g, _ = singular_locus()
    others = [u for u in range(L.U) if u not in g]
    idx = np.full((n, kmax), -1, dtype=np.int32)
    for r in range(n):
        if with_pair:
            pick = list(g) + rng.choice(others, int(rng.integers(0, kmax - 1)), replace=False).tolist()
        else:
            k = int(rng.integers(0, kmax + 1))
            pick = rng.choice(others, k, replace=False).tolist()
            if k and r % 2:
                pick[0] = g[r % 4 // 2]
        idx[r, :len(pick)] = sorted(pick)
    return idx


@pytest.mark.parametrize("kmax", [3, 6])
def test_singular_block_scoring(kmax):
    """kmax 3: the lane kernel (which hands such rows to the warp's mantissa/exponent code), kmax 6: the warp kernel."""
    from oracle import oracle as O
    L = singular_locus()[0]
    rng = np.random.default_rng(50 + kmax)
    good, bad = union_rows(rng, 64, kmax, False), union_rows(rng, 6, kmax, True)
    want_l, want = O.score_union_configs(as_oracle(L), good)
    with engine_for(L, max(kmax, 3)) as e:
        np.testing.assert_allclose(e.score_union_configs(good), want_l, rtol=1e-10, atol=0)
        assert_results_match(e.read(), want)
        for row in bad:
            e.reset()
            expect_error(PIPSORT_E_SINGULAR, "matrix is singular", e.score_union_configs, row[None])
        e.reset()
        expect_error(PIPSORT_E_SINGULAR, "matrix is singular", e.score_union_configs, np.concatenate([good, bad[:1]]))


def test_singular_block_given_configs():
    from oracle import oracle as O
    L, _, (i, j) = singular_locus()
    n0, N = int(L.num_snps[0]), L.N
    lo, hi = min(i, j), max(i, j)
    m = next(x for x in range(n0) if x not in (i, j))           # a third study-0 SNP
    bad = np.array([[lo, hi, -1, -1], [-1, lo, hi, n0 + 2], sorted([m, lo, hi]) + [-1]], dtype=np.int16)
    rng = np.random.default_rng(9)
    good = np.full((200, 4), -1, dtype=np.int16)
    for r in range(len(good)):
        pick = set(rng.choice(N, int(rng.integers(0, 5)), replace=False).tolist())
        if {i, j} <= pick:
            pick.discard(j)
        good[r, :len(pick)] = sorted(pick)
    rc, want = O.given_configs(as_oracle(L), good)
    assert rc == 0
    with engine_for(L, 3) as e:
        r = e.compute_total_likelihood_given_configs(good)
        assert r.n_configs == len(good)
        assert_results_match(r, want)
        for row in bad:
            e.reset()
            expect_error(PIPSORT_E_SINGULAR, "matrix is singular", e.score_given_configs, row[None])
