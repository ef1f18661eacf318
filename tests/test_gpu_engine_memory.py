"""Device memory of an engine: every buffer comes from the engine's arena or from the device's default memory pool and goes
back when the engine is destroyed; a request no device can satisfy leaves the engine as it was; nothing is allocated while
a pass is being captured into a CUDA graph.  The pool is read through the driver API (libcuda) after a device
synchronise."""
import ctypes as C

import numpy as np
import pytest

from conftest import (assert_results_match, dataset_paths, engine_for, exh_plan_env, oracle_locus, synth_as_oracle_locus,
                      synth_locus)

pytestmark = pytest.mark.gpu

CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7
PIPSORT_E_ARG, PIPSORT_E_CUDA = 1, 2
IDX = np.array([[-1, -1, -1], [7, -1, -1], [0, 7, -1], [1, 4, 9]], dtype=np.int32)


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


def locus_dict(SL):
    return dict(num_snps=SL.num_snps, sigma=np.concatenate([s.ravel() for s in SL.sigma]), z=np.concatenate(SL.z), d=SL.d,
                K=SL.K, snp_map=SL.snp_map, gamma=SL.gamma, sharing_param=SL.sharing_param)


def cycle(L, SL):
    """One of everything that allocates: engines of every kind, the growing buffers, call-local temporaries."""
    import pipsort_b200 as P
    from oracle import oracle as O
    with engine_for(L, 3) as e:
        r = e.compute_total_likelihood(3)
        assert r.n_configs == 268
        e.flush_l2()
        e.enumerate(3, 5)
        e.reset()
        e.score_union_configs(IDX[:2])
        e.score_union_configs(np.tile(IDX, (50, 1)))                 # a larger batch: the scratch grows
        e.compute_total_likelihood_given_configs(np.array([[0, 5, -1], [2, 7, 9]], dtype=np.int16))
        e.sss(1)
        e.sss(3)                                                      # more SNPs per row: the search buffers grow
    with engine_for(L, 3) as a, engine_for(L, 3) as b:
        n = a.total_ranks(3)
        a.reset(); b.reset()
        a.run_exhaustive(3, 0, n // 2); b.run_exhaustive(3, n // 2, n)
        a.merge_from(b)
        assert a.read().n_configs == 268
    ld_files, z_files, _, _ = dataset_paths("small_example")
    lds, zs = [O.read_ld(f) for f in ld_files], [O.read_z(f)[1] for f in z_files]
    with P.Engine(L.n_snps, lds, zs, L.d, 0.0, L.snp_map, gamma=L.gamma, sharing_param=L.p, max_causal=3, raw_ld=True) as e:
        e.compute_total_likelihood(3)
    P.preprocess_study(lds[0], zs[0])
    with engine_for(L, 8, prior_classes=True) as e:                    # its class-resolved store overflows the arena
        e.reset()
        e.run_exhaustive(3)
        e.read_prior_grid([(0.01, 0.75)])
        e.read_prior_grid([(0.01, p) for p in np.linspace(0.0, 1.0, 64)])   # the grid buffer grows
    SD = locus_dict(SL)
    P.posterior_exhaustive(SD["num_snps"], SD["sigma"], SD["z"], SD["d"], SD["K"], SD["snp_map"], 3)
    P.posterior_exhaustive_grid(SD["num_snps"], SD["sigma"], SD["z"], SD["d"], SD["K"], SD["snp_map"], 3, [(0.01, 0.75), (0.2, 0.25)])
    P.posterior_exhaustive_batch([SD] * 9, 3)


def test_engines_return_all_pool_memory(pool_used):
    """After one warm-up cycle, every further cycle leaves exactly as much of the pool in use as before it."""
    L = oracle_locus("small_example")
    SL = synth_locus(40, overlap=0.5, seed=77)
    cycle(L, SL)
    base = pool_used()
    for _ in range(2):
        cycle(L, SL)
        assert pool_used() == base


def test_refused_scratch_leaves_the_engine_usable(pool_used):
    """An engine that has scored a batch (its scratch holds it) is asked for a batch whose scratch no device can hold (2^40
    rows: 4 TB of indices): the call fails at once, and the engine keeps no freed buffer and no stale capacity: it scores
    the next batch as a fresh engine does, and destroy returns everything."""
    import pipsort_b200 as P
    L = oracle_locus("small_example")
    with engine_for(L, 3) as fresh:
        want_l = fresh.score_union_configs(IDX)
        want = fresh.read()
    base = pool_used()
    e = engine_for(L, 3)
    e.score_union_configs(IDX)                            # scratch for 4 rows: the refused call replaces it
    e.reset()
    lib = P.lib()
    assert lib.pipsort_score_union_configs(e._h, None, 1 << 40, 0, None, None) == PIPSORT_E_CUDA
    e.reset()
    np.testing.assert_array_equal(e.score_union_configs(IDX), want_l)
    got = e.read()
    assert got.n_configs == want.n_configs
    assert_results_match(got, want, rtol=1e-12)
    e.close()
    with engine_for(L, 3) as again:
        again.compute_total_likelihood(3)
    assert pool_used() == base


def test_capture_refuses_to_allocate():
    """Under a forced plan of one warp-step per chunk, far more descriptors than the engine's buffer holds: growing it
    inside a capture is refused with PIPSORT_E_ARG before anything is recorded, and the engine's next pass is right."""
    import pipsort_b200 as P
    from oracle import oracle as O
    SL = synth_locus(150)
    want = O.exhaustive(synth_as_oracle_locus(SL), 3)
    with engine_for(SL, 3) as e:
        e.compute_total_likelihood(3)
        with exh_plan_env(1):
            e.graph_begin()
            with pytest.raises(P.PipsortError) as err:
                e.run_exhaustive(3)
            e.graph_end()
        assert err.value.code == PIPSORT_E_ARG and "before capturing" in str(err.value)
        r = e.compute_total_likelihood(3)
    assert r.n_configs == want.n_eval
    assert_results_match(r, want)


def test_search_that_grows_its_hash_table(pool_used):
    """6000 SNPs per study (U = 7200), c = 3: the search needs room for up to 115,155 configurations in one round, so the
    explored-configuration table grows past its first 2^16 slots (to 2^18) and is rehashed on the way.  Every draw must
    still follow the oracle's, and destroy returns the tables to the pool."""
    from oracle import oracle as O
    from pipsort_b200 import synth
    SL = synth.make_locus(6000, overlap=0.8)
    want = O.sss(synth_as_oracle_locus(SL), 3, max_iter=20)
    seen, need = 0, 0                                     # the table is reserved for twice what a round may hold
    for _, nbd, new, _ in want.extra["trace"]:
        need, seen = max(need, seen + int(nbd)), seen + int(new)
    assert need == 115155                                 # 2 need > 2^17: 2^18 slots
    base = pool_used()
    with engine_for(SL, 3) as e:
        r, iters, why = e.sss(3, max_iterations=20)
    assert pool_used() == base
    assert iters == want.extra["n_iter"] == 8 and why == 1
    assert_results_match(r, want)
