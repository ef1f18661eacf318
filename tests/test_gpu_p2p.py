"""The peer-memory combine step (p2p.cuh: CUDA IPC mailboxes, system-scope fp64 atomics, device-side arrival / flow
control words) with TWO processes.  Both ranks use cuda:0 when the box has a single GPU -- CUDA IPC maps another
process's memory of the same device just as well, so export / connect / push / wait / merge / flow control all run for
real; with two GPUs the ranks take one each and the atomics cross NVLink.  gloo only carries the 64-byte handles."""
import os
import sys
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT, assert_results_match, engine_for, oracle_locus

pytestmark = pytest.mark.gpu


def _worker(rank, world, initfile, outdir):
    import faulthandler
    faulthandler.dump_traceback_later(120, exit=True)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from pipsort_b200 import distributed as D
    from oracle import oracle as O
    from conftest import golden
    dist.init_process_group("gloo", init_method=f"file://{initfile}", rank=rank, world_size=world)
    try:
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        L = oracle_locus("small_example")
        want = O.exhaustive(L, 3)
        Le = oracle_locus("example", p=0.25)
        with engine_for(L, 3, device=dev) as e, engine_for(Le, 2, device=dev) as e2:
            assert D.connect_p2p(e)
            assert D.connect_p2p(e2)
            for rep in range(5):                       # several epochs: arrivals / consumed flow control
                r = D.compute_total_likelihood_sharded(e, 3, collective="p2p")
                if rank == 0:
                    assert r.n_configs == want.n_eval == 268
                    assert_results_match(r, want)
                else:
                    assert r is None
            # lopsided caller-supplied split, and a locus whose log-likelihoods span thousands of nats (many bins)
            r = D.compute_total_likelihood_sharded(e, 3, bounds=[0, 5, e.total_ranks(3)], collective="p2p")
            if rank == 0:
                assert_results_match(r, want)
            r2 = D.compute_total_likelihood_sharded(e2, 2, collective="p2p")
            if rank == 0:
                assert r2.n_configs == 216817
                assert_results_match(r2, golden("example_c2_p025"))
            # the repeatable pass (what bench.py times): no reset between passes -- the push empties the senders, the root
            # sums the peers' slots inside its finalize (few bins) or merges + finalizes (tests/example: ~80 bins)
            for eng, cc, w in ((e, 3, want), (e2, 2, golden("example_c2_p025"))):
                eng.reset(); eng.sync()
                dist.barrier()
                b = eng.shard_ranks(cc, world)
                for rep in range(4):
                    D.pass_exhaustive_sharded(eng, cc, b, collective="p2p")
                    if rank == 0:
                        rr = eng.fetch()
                        assert rr.n_configs == (268 if cc == 3 else 216817)
                        assert_results_match(rr, w)
                eng.sync()
                dist.barrier()
                leftover = eng.read()                      # every rank's store is empty after a pass
                assert leftover.n_configs == 0 and leftover.total == 0.0 and not leftover.postValues.any()
                dist.barrier()
        open(os.path.join(outdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_two_ranks_combine_over_peer_memory():
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(2, os.path.join(tmp, "init"), tmp), nprocs=2, join=True)
        assert os.path.exists(os.path.join(tmp, "ok0")) and os.path.exists(os.path.join(tmp, "ok1"))


def _nccl_worker(rank, world, initfile, outdir):
    import faulthandler
    faulthandler.dump_traceback_later(45, exit=True)           # a hung collective must not hang the suite
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from pipsort_b200 import distributed as D
    from oracle import oracle as O
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"file://{initfile}", rank=rank, world_size=world,
                            device_id=torch.device(f"cuda:{rank}"))
    try:
        from conftest import golden
        L = oracle_locus("small_example")
        want = O.exhaustive(L, 3)
        Le = oracle_locus("example", p=0.25)
        # the engines stay on their OWN streams: the helpers must order the all-reduce after the kernels themselves
        with engine_for(L, 3, device=rank) as e, engine_for(Le, 2, device=rank) as e2:
            for rep in range(4):
                r = D.compute_total_likelihood_sharded(e, 3, collective="allreduce")
                assert r.n_configs == want.n_eval == 268
                assert_results_match(r, want)
                r2 = D.compute_total_likelihood_sharded(e2, 2, collective="allreduce")
                assert r2.n_configs == 216817
                assert_results_match(r2, golden("example_c2_p025"))
            # one SSS neighbourhood split over the ranks, accumulators rank-partial until read_sharded
            rng = np.random.default_rng(3)
            idx = np.full((40, 3), -1, dtype=np.int32)
            for i in range(1, 40):
                k = int(rng.integers(1, 4))
                idx[i, :k] = np.sort(rng.choice(L.U, k, replace=False))
            want_l, want_acc = O.score_union_configs(L, idx)
            e.reset()
            got_l = D.score_union_configs_sharded(e, idx)
            np.testing.assert_allclose(got_l, want_l, rtol=1e-10)
            assert_results_match(D.read_sharded(e), want_acc)
        open(os.path.join(outdir, f"ok{rank}"), "w").write("ok")
    except BaseException:
        import traceback
        traceback.print_exc()
        os._exit(1)
    # (no destroy_process_group: NCCL's communicator teardown blocks in this spawn + file-store setting on the 2-GPU box
    #  -- both ranks were seen waiting inside it after a green test body; the processes end here instead)
    torch.cuda.synchronize()
    sys.stdout.flush(); sys.stderr.flush()
    os._exit(0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="NCCL needs one GPU per rank")
def test_two_ranks_nccl_allreduce_without_stream_binding():
    """The NCCL path of distributed.py with engines left on their own streams (no bind_engine_to_current_stream)."""
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_nccl_worker, args=(2, os.path.join(tmp, "init"), tmp), nprocs=2, join=True)
        assert os.path.exists(os.path.join(tmp, "ok0")) and os.path.exists(os.path.join(tmp, "ok1"))


def _sss_worker(rank, world, initfile, outdir):
    import faulthandler
    faulthandler.dump_traceback_later(120, exit=True)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from pipsort_b200 import distributed as D
    from pipsort_b200 import synth
    from oracle import oracle as O
    from conftest import golden, args_to_params, synth_as_oracle_locus
    dist.init_process_group("gloo", init_method=f"file://{initfile}", rank=rank, world_size=world)
    try:
        dev = rank % torch.cuda.device_count()
        torch.cuda.set_device(dev)
        # the reference's own `-q 1` dumps: same trajectory (round count, stop reason), same accumulators
        for name in ("small_sss_c3_p075", "example_sss_c2_p025"):
            g = golden(name)
            prm = args_to_params(g["args"])
            L = oracle_locus(g["dataset"], p=prm["p"], gamma=prm["gamma"], s=prm["s"], t=prm["t"])
            want = O.sss(L, prm["c"])
            with engine_for(L, prm["c"], device=dev) as e:
                assert D.connect_p2p(e)
                for rep in range(2):                               # a second search on the same engine: epochs keep counting
                    r, iters, why = D.sss_sharded(e, prm["c"])
                    assert iters == want.extra["n_iter"]
                    assert (why == 1) == any("hit break condition" in f for f in g["stdout_flags"])
                    if rank == 0:
                        assert_results_match(r, g)
                    else:
                        assert r is None
        # the longest trajectory we found (9 rounds; 12+12 SNPs), against the oracle ...
        SL = synth.make_locus(12, overlap=0.7, seed=18)
        want = O.sss(synth_as_oracle_locus(SL), 3)
        assert want.extra["n_iter"] == 9
        with engine_for(SL, 3, device=dev) as e:
            assert D.connect_p2p(e)
            r, iters, why = D.sss_sharded(e, 3)
            assert iters == 9 and why == 1
            if rank == 0:
                assert_results_match(r, want)
            # ... and with the convergence rule switched on from round 2 (the reference starts at round 100, which this search
            # never reaches): the running total every rank consults is the sum over ALL ranks' partial accumulators, so
            # the split search must stop in the same round with the same accumulators as the search on one GPU
            os.environ["PIPSORT_SSS_CONV_FROM"] = "2"
            try:
                one, it1, why1 = e.sss(3)
                r, iters, why = D.sss_sharded(e, 3)
            finally:
                os.environ.pop("PIPSORT_SSS_CONV_FROM", None)
            assert (iters, why) == (it1, why1) and why1 == 2 and it1 < 9
            if rank == 0:
                assert_results_match(r, one, rtol=1e-12)
        open(os.path.join(outdir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sss_neighbourhoods_split_over_ranks(world):
    """pipsort_sss_sharded: every rank scores its share of each round's unseen neighbours, the values travel through the
    peer-memory mailboxes, the replicated search state follows the reference's trajectory on every rank."""
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_sss_worker, args=(world, os.path.join(tmp, "init"), tmp), nprocs=world, join=True)
        assert all(os.path.exists(os.path.join(tmp, f"ok{r}")) for r in range(world))
