#!/usr/bin/env python
"""bench.py -- causal configurations / second of the exhaustive posterior calculation (BASELINE.json metric).

A "step" is one pass of the hot path (PostCal::computeTotalLikelihood, postcal.cpp:716-1092) over one
synthetic locus: enumerate + score every union subset of size <= c in this rank's shard of the rank space,
combine the accumulator stores of all ranks over NVLink peer memory (engine kernels; NCCL all-reduce as the
fallback), finalize (bins -> log-space results).  The reset of the accumulators and the re-arming of the work
queue are folded into the kernels that touch them last, so a pass is 2 launches on one GPU.

  value     whole-job configurations/s with the locus already resident in HBM, device-timed (CUDA events on
            the stream everything is launched on), max over ranks
  e2e       the same metric through the public API with HOST buffers: engine creation (H2D of LD / z / maps),
            the pass, and the D2H read of the result arrays inside the timed region -- the batch call over
            distinct loci (headline) and the single-locus call (e2e.single_locus_call)
  roofline  FP64 vector-pipe roofline of the dominant kernel (the size-c class launch): algorithmic flops
            (SURVEY.md 8d formula, counted exactly by class) / its device time / the DFMA peak measured here;
            traffic = DRAM bytes of one launch from the ncu capture of this build (profiles/traffic.json)
  cpu_baseline   the reference's own OpenMP CPU build (oracle/_ref/PIPSORT, unmodified sources) on this host,
            on a bounded sample of the same workload (the size <= 2 prefix of the rank space, `-c 2`);
            falls back to the OpenMP port of the oracle when the reference binary is not present
  side keys (same line): saturating (1500 SNPs/study, c=3), A300c2_p0.25 / A300c2_p0.75 (BASELINE.json configs[2]),
            D5000c5_sss (configs[4]: one shotgun-search neighbourhood at 5000 SNPs/study, c=5, with FP64 roofline
            fraction and LD-gather GB/s against the measured HBM bandwidth)

python bench.py --impl reference ... times only the reference CPU implementation and prints the same line.
python bench.py --dump-outputs DIR ... also writes the result arrays of the last timed pass as DIR/<name>.npy (float64);
the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (SNPs per study, overlap, c)   -- BASELINE.json configs[3] / configs[2] / the saturating B10 of SURVEY 8d
    "B150c3": (150, 0.8, 3),
    "A300c2": (300, 0.8, 2),
    "B1500c3": (1500, 0.8, 3),
}
def traffic_for(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, as `profiles/summarize.py --traffic`
    extracted it from the `ncu --set full` capture of the build that is benchmarked (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            ent = json.load(f).get(workload)
        return (int(ent["bytes"]), ent["source"]) if ent else (None, None)
    except Exception:
        return None, None


METRIC = "causal configurations/sec (exhaustive, c=3, synthetic 150-SNP/study two-ancestry locus)"
UNIT = "configs/s"


def class_flops(snp_map, c):
    """(algorithmic flops, configurations) of the size-c class and of the whole run (SURVEY.md 8d)."""
    from pipsort_b200 import synth
    tot, ntot = synth.flops_per_config_total(snp_map, c)
    low, nlow = synth.flops_per_config_total(snp_map, c - 1) if c > 0 else (0.0, 0)
    return (tot - low, ntot - nlow), (tot, ntot)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            with open(self.path) as f:
                for line in f:
                    t = [x.strip() for x in line.split(",")]
                    if len(t) < 9:
                        continue
                    try:
                        sm.append(float(t[1])); mx.append(float(t[2]))
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), t[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------
# CPU arms (test infrastructure: the only place bench.py executes anything under oracle/)
# ---------------------------------------------------------------------------------------------------------
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "PIPSORT")


def reference_cpu_run(L, c_sample, workdir):
    """One run of the UNMODIFIED reference CLI (exhaustive, `-c c_sample`) on the locus; returns
    (configurations, seconds of its own 'Time to eval all' timer, wall seconds)."""
    from pipsort_b200 import synth
    ld, z, mp, ns = synth.write_files(L, os.path.join(workdir, "in"))
    env = dict(os.environ, OPENBLAS_NUM_THREADS="1")
    t = time.time()
    p = subprocess.run([REF_BIN, "-l", ld, "-z", z, "-m", mp, "-n", ns, "-o", os.path.join(workdir, "out"), "-c",
                        str(c_sample), "-g", repr(L.gamma), "-p", repr(L.sharing_param)], capture_output=True,
                       text=True, env=env, cwd=workdir)
    wall = time.time() - t
    if p.returncode != 0:
        raise RuntimeError("reference CLI failed: " + p.stderr[-500:])
    m = re.search(r"Time to eval all=\s*(\d+)\[", p.stdout)
    secs = int(m.group(1)) * 1e-6 if m else wall
    return synth.count_configs(L.snp_map, c_sample), secs, wall


def port_cpu_run(L, c, seconds_target=10.0):
    """OpenMP port of the oracle on a rank sub-range sized to ~seconds_target; returns (configs, seconds, cores)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from conftest import synth_as_oracle_locus
    from oracle import oracle as O
    OL = synth_as_oracle_locus(L)
    cores = os.cpu_count() or 1
    tot = O.total_union_subsets(OL.U, c)
    n = min(tot, 20000)
    lo = tot - n                                  # the size-c class dominates; sample from its end
    t = time.time(); _, ne = O.exhaustive_omp(OL, c, lo, tot, cores); dt = time.time() - t
    if dt < seconds_target / 4 and n < tot:       # scale the sample up once
        n = int(min(tot, n * seconds_target / max(dt, 1e-3)))
        lo = tot - n
        t = time.time(); _, ne = O.exhaustive_omp(OL, c, lo, tot, cores); dt = time.time() - t
    return ne, dt, cores, f"union-subset ranks [{lo},{tot}) of {tot}"


def cpu_baseline(L, c):
    cores = os.cpu_count() or 1
    if os.path.exists(REF_BIN):
        try:
            with tempfile.TemporaryDirectory() as tmp:
                n, secs, wall = reference_cpu_run(L, c - 1, tmp)
            return {"value": n / secs, "unit": UNIT, "cores": cores, "kind": "reference",
                    "sample": f"unmodified reference CLI `-c {c - 1}` on the same locus = the size<={c - 1} prefix of the "
                              f"rank space ({n} configurations); its own 'Time to eval all' {secs:.2f} s (wall {wall:.2f} s); "
                              f"the reference forces 64 OpenMP threads (postcal.cpp:748) on {cores} host cores"}
        except Exception as ex:  # fall through to the port
            err = str(ex)[:200]
    else:
        err = "oracle/_ref/PIPSORT not built"
    ne, dt, cores, what = port_cpu_run(L, c)
    return {"value": ne / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"OpenMP port of the oracle (closed-form O(k^3) likelihood), {what}, {ne} configurations in {dt:.2f} s ({err})"}


def run_reference_arm(args, L, c, wl):
    """bench.py --impl reference: rank 0 alone times the reference's own CPU implementation."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    vals, walls = [], []
    kind = "reference" if os.path.exists(REF_BIN) else "port"
    sample = ""
    for i in range(args.warmup + args.steps):
        timed = i >= args.warmup
        if kind == "reference":
            with tempfile.TemporaryDirectory() as tmp:
                n, secs, wall = reference_cpu_run(L, c - 1, tmp)
            sample = (f"unmodified reference CLI `-c {c - 1}` = size<={c - 1} prefix of the rank space, {n} configurations per step; "
                      f"64 OpenMP threads forced by the reference on {cores} cores; timed with its own 'Time to eval all'")
        else:
            n, secs, cores, what = port_cpu_run(L, c)
            sample = f"oracle OpenMP port, {what}"
        if timed:
            vals.append(n / secs); walls.append(secs)
    v = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
            "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(walls)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl_desc(wl, L, c), "l2": "n/a (CPU)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


def wl_desc(wl, L, c):
    sh, o0, o1 = L.n_types()
    return (f"{wl}: synthetic two-ancestry locus, {int(L.num_snps[0])}+{int(L.num_snps[1])} SNPs, U={L.U} "
            f"({sh} shared, {o0}+{o1} study-specific), exhaustive c={c}, p={L.sharing_param}, gamma={L.gamma}, seed 20261018")


# ---------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def claim_stdout():
    """ONE JSON line on stdout is the contract, but libraries print there too (NCCL's version banner at communicator
    creation, for instance): point fd 1 at stderr for the whole run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def dump_outputs(res, outdir):
    """What a caller of the timed pass receives (the pipsort_b200.Results of the last timed step): one float64 array
    per result member.  Only rank 0 calls it: with several GPUs the root holds the whole job's result."""
    os.makedirs(outdir, exist_ok=True)
    arrays = {"total": [res.total], "postValues": res.postValues, "noCausal": res.noCausal, "sharedPips": res.sharedPips,
              "sharedLL": res.sharedLL, "notSharedLL": res.notSharedLL, "n_configs": [res.n_configs]}
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="B150c3", choices=sorted(WORKLOADS))
    ap.add_argument("--collective", default="p2p", choices=["p2p", "allreduce"],
                    help="multi-GPU combine step: the engine's peer-memory kernels (default) or one NCCL all-reduce")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sat", action="store_true", help="skip the saturating B1500c3 side measurement")
    ap.add_argument("--no-side", action="store_true", help="skip the A300c2 / D5000c5 side measurements (BASELINE.json configs[2], [4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result arrays of the last timed pass as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm only times the CPU implementation")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from pipsort_b200 import synth
    n_per, overlap, c = WORKLOADS[args.workload]
    L = synth.make_locus(n_per, overlap=overlap)
    if args.impl == "reference":
        run_reference_arm(args, L, c, args.workload)
        return

    import torch
    import torch.distributed as dist
    import pipsort_b200 as P
    from pipsort_b200 import distributed as D

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")
    # everything (engine kernels, NCCL all-reduce, timing events) is enqueued on ONE non-default stream
    work_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(work_stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    collective_used = []
    graph_used = []
    hbm_gbs = 6548.2
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm_gbs = float(json.load(f).get("hbm_gbs", hbm_gbs))
    except Exception:
        pass

    def measure(L, c, steps, warmup, clocks=False):
        """Device-timed passes on the resident locus.  A pass = this rank's exhaustive launch + the combine step + the
        finalize; the reset of the accumulators is folded into the kernels that read them last."""
        total_configs = synth.count_configs(L.snp_map, c)
        e = P.Engine(L.num_snps, L.sigma, L.z, L.d, L.K, L.snp_map, gamma=L.gamma, sharing_param=L.sharing_param,
                     max_causal=c, device=local)
        stream = torch.cuda.current_stream()
        e.set_stream(stream.cuda_stream)
        b = e.shard_ranks(c, world)
        # combine step: the engine's own peer-memory kernels over NVLink (CUDA IPC mailboxes) when the ranks can map each
        # other, else ONE NCCL all-reduce(sum) of the accumulator store
        coll = "allreduce"
        if world > 1 and args.collective != "allreduce":
            coll = "p2p" if D.connect_p2p(e) else "allreduce"
        collective_used.append(coll)

        def step():
            D.pass_exhaustive_sharded(e, c, b, collective=coll)

        e.reset()
        e.flush_l2(); step()                  # first pass: builds the pair tables, uploads the work plan
        l0 = e.launch_count()
        e.flush_l2(); step()
        launches_per_step = e.launch_count() - l0
        # the pass is a fixed sequence of the engine's launches: record it once into a CUDA graph and replay it with one
        # launch per step.  The NCCL fallback is issued by torch and stays un-captured.
        run = step
        graphed = False
        if coll != "allreduce" or world == 1:
            e.graph_begin(); step(); gid = e.graph_end()
            run = lambda: e.graph_launch(gid)   # noqa: E731
            graphed = True
        graph_used.append(graphed)
        for _ in range(warmup):
            e.flush_l2(); run()
        sampler = ClockSampler(local)
        if clocks and rank == 0:
            sampler.start()                   # before the barrier: spawning nvidia-smi must not delay rank 0's first steps
        barrier()
        evs = []
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t_wall = time.perf_counter()
        for a, z in pairs:
            e.flush_l2()                      # L2 flushed between timed iterations (outside the event pair)
            a.record(stream); run(); z.record(stream)
            evs.append((a, z))
        barrier()
        t_wall = time.perf_counter() - t_wall
        res = e.fetch() if rank == 0 else None            # the last timed pass: the whole job's result on the root
        if clocks:
            # the timed region lasts a few milliseconds: keep the SAME step running back to back for another ~0.3 s,
            # untimed, so that nvidia-smi (20 ms period) sees the clocks / throttle reasons under this load
            t_load = time.perf_counter()
            while time.perf_counter() - t_load < 0.3:
                for _ in range(50):
                    run()
                e.sync()
            barrier()
        clk = sampler.stop() if clocks and rank == 0 else None
        if clk is not None:
            clk["window"] = "timed region + 0.3 s of the same step repeated back to back (untimed), nvidia-smi every 20 ms"
        ms = [a.elapsed_time(z) for a, z in evs]
        if os.environ.get("PIPSORT_BENCH_DEBUG"):
            print(f"[rank {rank}] per-step ms: " + " ".join(f"{x:.4f}" for x in ms), file=sys.stderr, flush=True)
        # dominant-kernel duration: a few extra passes timed on the launch itself (CUDA events around the kernel)
        kms = []
        for _ in range(min(max(steps, 3), 10)):
            e.flush_l2(); step(); kms.append(e.last_kernel_ms())
        tot_ms = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
        k_ms = torch.tensor([float(np.mean(kms))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(k_ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        e.close()
        if rank == 0:
            assert res.n_configs == total_configs, (res.n_configs, total_configs)
        return dict(total_configs=total_configs, ms_per_step=float(tot_ms.item()) / steps, kernel_ms=float(k_ms.item()),
                    launches=launches_per_step * steps, launches_per_step=launches_per_step,
                    wall_ms_per_step=1e3 * t_wall / steps, timed_region_s=float(tot_ms.item()) * 1e-3, clocks=clk, result=res)

    def roofline_of(L, c, m, peak, workload=None):
        (cf, cn), _ = class_flops(L.snp_map, c)
        achieved = cf / world / (m["kernel_ms"] * 1e-3) / 1e12     # the launch on rank r covers 1/world of the class
        tr, src = traffic_for(workload) if (workload and world == 1) else (None, None)
        r = {"bound": "fp64", "achieved": achieved, "peak": peak / 1e12, "unit": "TFLOP/s", "frac": achieved / (peak / 1e12),
             "traffic": tr, "kernel_ms": m["kernel_ms"], "flop_per_launch": cf / world, "flop_per_config": cf / max(cn, 1)}
        if src:
            r["traffic_source"] = src
        return r

    def measure_e2e(L, c, steps, warmup):
        """Public API with HOST (pinned) buffers: create (H2D) + pass + read (D2H) + destroy, wall clock between syncs."""
        total_configs = synth.count_configs(L.snp_map, c)
        sig = torch.from_numpy(np.concatenate([s.ravel() for s in L.sigma])).pin_memory()
        z = torch.from_numpy(np.concatenate(L.z)).pin_memory()
        h2d = sig.numel() * 8 + z.numel() * 8 + L.snp_map.size * 4 * 3 + 2 * 16
        d2h = 8 * (1 + 2 + L.N + 3 * L.U)
        sig_np, z_np = sig.numpy(), z.numpy()

        # (a) ONE locus per call.  N = 1: pipsort_posterior_exhaustive.  N > 1: the same locus with its rank space sharded
        # over the GPUs and the stores combined over peer memory -- every rank creates its engine from host buffers,
        # the root reads the result.
        def once():
            if world == 1:
                return P.posterior_exhaustive(L.num_snps, sig_np, z_np, L.d, L.K, L.snp_map, c, gamma=L.gamma,
                                              sharing_param=L.sharing_param, device=local)
            e = P.Engine(L.num_snps, sig_np, z_np, L.d, L.K, L.snp_map, gamma=L.gamma,
                         sharing_param=L.sharing_param, max_causal=c, device=local)
            coll = "p2p" if (args.collective != "allreduce" and D.connect_p2p(e)) else "allreduce"
            if coll == "allreduce":
                D.bind_engine_to_current_stream(e)
            r = D.compute_total_likelihood_sharded(e, c, collective=coll)
            e.close()                     # (mailboxes and peer mappings belong to the process: nothing to wait for)
            return r

        for _ in range(warmup):
            once()
        barrier()
        t = time.perf_counter()
        for _ in range(steps):
            r = once()
        barrier()
        dt = torch.tensor([time.perf_counter() - t], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        serial_ms = 1e3 * float(dt.item()) / steps
        # (b) the call a user with many loci makes -- a LIST of loci in one C-ABI call (pipsort_posterior_exhaustive_batch).
        # Every step (= locus) has its OWN pinned host arrays (distinct objects: nothing is shared or memoised between
        # loci), its own pinned-host -> device copy of the LD matrices / z / maps, its own kernels and its own device ->
        # host read of the result arrays inside the timed region; the engine overlaps the uploads and preparation of locus
        # i+1 and the read-back of locus i-1 with the evaluation of locus i (three streams).  With several GPUs the LOCI
        # are dealt out to the ranks (independent units, no collective): every rank runs the same call on its own list.
        nb = max(steps, 8) * 4
        loci = []
        for i in range(nb):
            sg = sig.clone().pin_memory(); zz = z.clone().pin_memory()
            loci.append(dict(num_snps=L.num_snps.copy(), sigma=sg.numpy(), z=zz.numpy(), d=L.d.copy(), K=L.K,
                             snp_map=L.snp_map.copy(), gamma=L.gamma, sharing_param=L.sharing_param, _keep=(sg, zz)))
        P.posterior_exhaustive_batch(loci[:8], c, device=local)
        # the timed region is the C-ABI call (pipsort_posterior_exhaustive_batch) and nothing else: the argument block
        # (arrays of pipsort_locus / pipsort_outputs structs pointing at the pinned host arrays) is built beforehand, the
        # result buffer is sliced afterwards -- Python marshalling (~30 us per locus) is not part of the engine
        batch = P.LocusBatch(loci, c, device=local)
        # the call lasts a few milliseconds of host wall clock: it is repeated BATCH_REPS times and the mean is reported
        # (a single sample moved by +-40 % from run to run)
        BATCH_REPS = 5
        for _ in range(2):                # warm-up calls: the first full-size call creates the streams, events and pinned
            batch.run()                   # staging buffers of its nine engines in flight (0.26 ms per locus against 0.045)
        barrier()
        t = time.perf_counter()
        per_call = []
        for _ in range(BATCH_REPS):
            tc = time.perf_counter()
            batch.run()
            per_call.append(1e3 * (time.perf_counter() - tc) / nb)
        barrier()
        if os.environ.get("PIPSORT_BENCH_DEBUG"):
            print(f"[rank {rank}] batch call, ms per locus: " + " ".join(f"{x:.4f}" for x in per_call), file=sys.stderr, flush=True)
        dtb = torch.tensor([time.perf_counter() - t], dtype=torch.float64, device=dev)
        rs = batch.results()
        if world > 1:
            dist.all_reduce(dtb, op=dist.ReduceOp.MAX)
        dtb = float(dtb.item()) / BATCH_REPS
        assert all(x.n_configs == total_configs for x in rs)
        if r is not None:
            assert abs(rs[-1].total - r.total) <= 1e-9 * abs(r.total)
        return {"value": total_configs * nb * world / dtb, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": 1e3 * dtb / (nb * world), "what": "batch call (loci_per_call distinct loci per rank in ONE C-ABI call)",
                "loci_per_call": nb, "loci_total": nb * world, "calls_timed": BATCH_REPS, "calls_warmup": 2,
                "single_locus_call": {"value": total_configs / (serial_ms * 1e-3), "unit": UNIT, "ms_per_step": serial_ms,
                                      "what": ("one locus per C-ABI call (create + pass + read + destroy)" if world == 1 else
                                               "one locus per call, its rank space sharded over the GPUs, stores combined over peer "
                                               "memory, result read on the root (create + pass + combine + read + destroy on every rank)")},
                "timing": "host wall clock (max over ranks) around ONE C-ABI call per rank (pipsort_posterior_exhaustive_batch; argument "
                          "structs built before, results sliced after) that evaluates loci_per_call DISTINCT loci "
                          "(own pinned host arrays each) -- per locus: H2D of LD / z / maps, preparation + exhaustive + finalize "
                          "kernels, D2H of the result arrays; three loci in flight on three streams per GPU; loci dealt out to "
                          "the ranks, no collective"}

    def measure_sss(peak):
        """BASELINE.json configs[4]: one neighbourhood of the stochastic shotgun search on the 5000-SNP/study locus (c = 5;
        29,984 union configurations x up to 3^5 expansions) through pipsort_score_union_configs_device -- the launch the
        search issues once per round (sss_postcal.cpp:223-255) -- and the whole search through pipsort_sss.  With N GPUs
        the neighbourhood list is cut into N slices (distributed.score_union_configs_sharded_device): every rank scores
        its slice, the max-|l| values are all-gathered."""
        Ld = synth.make_locus(5000, overlap=0.8)
        U, cc = Ld.U, 5
        cur = sorted({int(np.where(Ld.snp_map[0] == int(np.argmax(np.abs(Ld.z[0]))))[0][0]), 17, U // 2 - 1, U - 2})
        non = np.array([g for g in range(U) if g not in set(cur)], dtype=np.int32)
        rows = []
        for g in non:                                     # zero: added SNP outer, dropped position inner (sss_postcal.cpp:72-99)
            for m in range(len(cur)):
                rows.append(sorted(cur[:m] + cur[m + 1:] + [int(g)]))
        rows += [cur[:m] + cur[m + 1:] for m in range(len(cur))]
        rows += [sorted(cur + [int(g)]) for g in non]
        idx = np.full((len(rows), cc), -1, dtype=np.int32)
        for i, v in enumerate(rows):
            idx[i, :len(v)] = v
        t0 = time.perf_counter()
        e = P.Engine(Ld.num_snps, Ld.sigma, Ld.z, Ld.d, Ld.K, Ld.snp_map, gamma=Ld.gamma, sharing_param=Ld.sharing_param,
                     max_causal=cc, device=local)
        e.sync()
        create_s = time.perf_counter() - t0
        stream = torch.cuda.current_stream()
        e.set_stream(stream.cuda_stream)
        bnd = D.slice_bounds(len(rows), world)
        lo, hi = bnd[rank], bnd[rank + 1]
        d_idx = torch.from_numpy(idx[lo:hi].copy()).to(dev)
        width = max(bnd[r + 1] - bnd[r] for r in range(world))
        d_out = torch.zeros(width, dtype=torch.float64, device=dev)
        d_all = torch.empty(world * width, dtype=torch.float64, device=dev) if world > 1 else None

        def one(gather):
            e.score_union_configs_device(d_idx.data_ptr(), hi - lo, cc, 0, d_out.data_ptr())
            if gather:
                dist.all_gather_into_tensor(d_all, d_out)

        def timed(gather):
            for _ in range(3):
                one(gather)
            e.sync(); e.reset(); barrier()
            reps = 10
            evp = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for a, z in evp:
                a.record(stream); one(gather); z.record(stream)
            barrier()
            t_ms = torch.tensor([float(np.mean([a.elapsed_time(z) for a, z in evp]))], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
            return float(t_ms.item())

        ms = timed(False)                       # scoring launch of this rank's slice, max over ranks
        ms_nccl = timed(True) if world > 1 else None
        sh = (Ld.snp_map[0] >= 0) & (Ld.snp_map[1] >= 0)
        n_exp, flops, gather = 0, 0.0, 0
        for v in rows:
            a_sh = int(sh[v].sum()) if len(v) else 0
            f, n = synth.flops_of_union_subset(a_sh, int((Ld.snp_map[0][v] >= 0).sum()) - a_sh if len(v) else 0,
                                               int((Ld.snp_map[1][v] >= 0).sum()) - a_sh if len(v) else 0)
            flops += f; n_exp += n
            k0, k1 = int((Ld.snp_map[0][v] >= 0).sum()) if len(v) else 0, int((Ld.snp_map[1][v] >= 0).sum()) if len(v) else 0
            gather += 8 * (k0 * k0 + k1 * k1)
        # the whole search (device-resident search state; with N GPUs: pipsort_sss_sharded -- every round's neighbourhood
        # split over the ranks, the values exchanged through the peer-memory mailboxes): host wall clock, max over ranks
        sss = None
        e.set_stream(0)
        if world == 1 or D.connect_p2p(e):
            for rep in range(2):
                barrier()
                t1 = time.perf_counter()
                rs, it, why = D.sss_sharded(e, cc)
                dt = torch.tensor([time.perf_counter() - t1], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            if rank == 0:
                dtv = float(dt.item())
                sss = {"rounds": it, "stop_reason": why, "configs": rs.n_configs, "ms_total": 1e3 * dtv, "ms_per_round": 1e3 * dtv / max(it, 1),
                       "what": "pipsort_sss" if world == 1 else "pipsort_sss_sharded + combine over peer memory + read on the root"}
        if world > 1:
            dist.barrier()
        e.close()
        return {"workload": f"D5000c5_sss: synthetic 5000+5000 SNPs, U={U}, c=5; ONE neighbourhood of a 4-SNP state = {len(rows)} union "
                            f"configurations, {n_exp} expanded configurations, sliced over {world} GPU(s)",
                "ms_per_neighbourhood": ms, "value": n_exp / (ms * 1e-3), "unit": UNIT,
                "ms_with_nccl_allgather_of_the_values": ms_nccl,
                "union_configs_per_s": len(rows) / (ms * 1e-3),
                "roofline": {"bound": "fp64", "achieved": flops / (ms * 1e-3) / 1e12, "peak": peak / 1e12, "unit": "TFLOP/s",
                             "frac": flops / (ms * 1e-3) / peak, "flop_per_launch": flops,
                             "note": "algorithmic flops, SURVEY.md 8d phi(k) count per expanded configuration"},
                "ld_gather": {"bytes": gather, "gbs": gather / (ms * 1e-3) / 1e9, "hbm_peak_gbs": hbm_gbs,
                              "frac": gather / (ms * 1e-3) / 1e9 / hbm_gbs,
                              "note": "algorithmic gather: the k x k causal sub-blocks of both studies per union configuration, 8-byte "
                                      "words, from the 400 MB of HBM-resident LD"},
                "l2": "not flushed: the LD (400 MB) exceeds L2 (126 MB); launches back to back, as the search issues them",
                "create_s": create_s, "search": sss}

    peak = P.measure_fp64_peak(local)                      # FLOP/s, DFMA chains on every SM
    main_m = measure(L, c, args.steps, args.warmup, clocks=True)
    e2e = measure_e2e(L, c, max(3, min(args.steps, 10)), 2)
    value = main_m["total_configs"] / (main_m["ms_per_step"] * 1e-3)
    roof = roofline_of(L, c, main_m, peak, args.workload)
    roof["note"] = ("FP64 vector pipe (DFMA), no tensor cores / not HBM bound; achieved = ALGORITHMIC flops of the size-c class "
                    f"({roof['flop_per_launch']:.4g} flop, {roof['flop_per_config']:.1f}/configuration, SURVEY.md 8d) per launch / its "
                    f"CUDA-event duration ({main_m['kernel_ms']:.4f} ms); peak = DFMA micro-benchmark measured in this run "
                    "(MEASURED_PEAKS.json has no FP64 figure; nominal 37 TFLOP/s). The kernel shares Cholesky work between the "
                    "expansions of a union subset and skips, at compile time, the expansions a segment of SNPs of one study cannot "
                    "have, so it executes ~5x fewer flops than the algorithmic count: frac exceeds 1 on saturating loci; the "
                    "executed FP64 pipe utilisation (ncu) is in profiles/.")
    side = {}
    if args.workload == "B150c3" and not args.no_sat:
        Ls = synth.make_locus(1500, overlap=0.8)
        sm = measure(Ls, 3, 3, 3)
        side["saturating"] = {"workload": wl_desc("B1500c3", Ls, 3), "configs": sm["total_configs"], "ms_per_step": sm["ms_per_step"],
                              "value": sm["total_configs"] / (sm["ms_per_step"] * 1e-3), "unit": UNIT,
                              "roofline": roofline_of(Ls, 3, sm, peak, "B1500c3")}
    if args.workload == "B150c3" and not args.no_side:
        # BASELINE.json configs[2]: 300 SNPs/study, 80 % overlap, c = 2, p = 0.25 and 0.75, at this run's N
        for pv in (0.25, 0.75):
            La = synth.make_locus(300, overlap=0.8, sharing_param=pv)
            am = measure(La, 2, 5, 3)
            side[f"A300c2_p{pv}"] = {"workload": wl_desc("A300c2", La, 2), "configs": am["total_configs"], "ms_per_step": am["ms_per_step"],
                                     "value": am["total_configs"] / (am["ms_per_step"] * 1e-3), "unit": UNIT,
                                     "roofline": roofline_of(La, 2, am, peak, "A300c2")}
        side["D5000c5_sss"] = measure_sss(peak)            # BASELINE.json configs[4]
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(main_m["result"], args.dump_outputs)
        cpu = None
        if not args.no_cpu and world == 1:
            cpu = cpu_baseline(L, c)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": main_m["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": wl_desc(args.workload, L, c), "configs_per_step": main_m["total_configs"],
                           "l2": "flushed between timed steps (256 MiB memset outside the per-step event pair)",
                           "launch": (f"one CUDA-graph launch per step ({main_m['launches_per_step']} kernels recorded once: exhaustive"
                                      + (" + combine" if world > 1 else "") + " + finalize; accumulator reset and work-queue re-arm are "
                                      "folded into those kernels)" if graph_used and graph_used[0] else "individual launches"),
                           "sharding": (f"rank space split into {world} work-weighted contiguous ranges; combine step per step: "
                                        + ("non-root ranks write their accumulator stores into the root's memory over NVLink "
                                           "(engine kernels, CUDA IPC peer memory, self-validating words)"
                                           if collective_used and collective_used[0] == "p2p" else
                                           "one NCCL all-reduce(sum) of the accumulator store")) if world > 1 else "single GPU"},
                "clocks": main_m["clocks"], "e2e": e2e, "gpu_launches": main_m["launches"], "roofline": roof,
                "locus_wall_ms": e2e["ms_per_step"], "wall_ms_per_step": main_m["wall_ms_per_step"],
                "timed_region_s": main_m["timed_region_s"]}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        line.update(side)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
