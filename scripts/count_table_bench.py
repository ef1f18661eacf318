"""Cost of the count table (PIPSORT_CAUSAL_COUNTS), at c = 3:
  * kernel time (CUDA events around the exhaustive launch, L2 flushed before each launch) of the three instantiations of the
    exhaustive kernel -- ordinary store, class-resolved store, class-resolved store with the count table -- on the synthetic
    150- and 1500-SNP/study loci, the arms interleaved within each repetition; median and minimum over the repetitions;
  * ms per locus of the class-table batch (pipsort_class_evidence_batch) against the count-table batch
    (pipsort_count_table_batch) on 40 loci of 150 SNPs per study and 4 loci of 1500, synchronous calls, interleaved, median.
The count tables are checked against the class tables of the same loci (log-sum-exp over b0, 1e-12 relative).  The card's
name and power limit are read in the same run.
python scripts/count_table_bench.py [--reps N] [--out file.json]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from grid_batch_bench import as_dict, gpu_info  # noqa: E402
import pipsort_b200 as P  # noqa: E402
from pipsort_b200 import synth  # noqa: E402

ARMS = {"ordinary": {}, "classes": {"prior_classes": True}, "counts": {"causal_counts": True}}


def kernel_times(n_snps, reps):
    SL = synth.make_locus(n_snps)
    engines = {k: P.Engine(SL.num_snps, SL.sigma, SL.z, SL.d, SL.K, SL.snp_map, gamma=SL.gamma, sharing_param=SL.sharing_param,
                           max_causal=3, **kw) for k, kw in ARMS.items()}
    try:
        for e in engines.values():       # warm-up: module load, pair tables, plan
            for _ in range(2):
                e.reset(); e.run_exhaustive(3); e.last_kernel_ms()
        t = {k: [] for k in engines}
        for _ in range(reps):
            for k, e in engines.items():
                e.reset(); e.flush_l2(); e.run_exhaustive(3); t[k].append(e.last_kernel_ms())
        cnt = engines["counts"].read_count_table(3)
        np.testing.assert_allclose(P.class_tables_from_counts(cnt, 3), engines["classes"].read_class_evidence(3), rtol=1e-12, atol=0)
    finally:
        for e in engines.values():
            e.close()
    med = {k: float(np.median(v)) for k, v in t.items()}
    return {"snps_per_study": n_snps, "reps": reps, "kernel_ms": med, "kernel_ms_min": {k: float(np.min(v)) for k, v in t.items()},
            "counts_over_classes": med["counts"] / med["classes"], "counts_over_ordinary": med["counts"] / med["ordinary"]}


def batch_times(n_snps, n_loci, reps, seed):
    loci = [as_dict(synth.make_locus(n_snps, seed=seed + i)) for i in range(n_loci)]
    arms = {"class_tables": P.LocusBatch(loci, 3, class_evidence=True), "count_tables": P.LocusBatch(loci, 3, count_table=True)}
    for b in arms.values():
        for _ in range(2):
            b.run()
    t = {name: [] for name in arms}
    for _ in range(reps):
        for name, b in arms.items():
            t0 = time.perf_counter()
            b.run()
            t[name].append(1e3 * (time.perf_counter() - t0) / n_loci)
    np.testing.assert_allclose(P.class_tables_from_counts(arms["count_tables"].tables(), 3), arms["class_tables"].tables(),
                               rtol=1e-12, atol=0)
    return {"snps_per_study": n_snps, "loci": n_loci, "reps": reps,
            "ms_per_locus": {name: float(np.median(v)) for name, v in t.items()},
            "ms_per_locus_min": {name: float(np.min(v)) for name, v in t.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=0, help="repetitions (default 30 for 150 SNPs/study, 5 for 1500)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"gpu": gpu_info(), "c": 3, "kernel": [], "batch": []}
    print(json.dumps({"gpu": out["gpu"]}), flush=True)
    for n_snps, reps in ((150, a.reps or 30), (1500, a.reps or 5)):
        rec = kernel_times(n_snps, reps)
        out["kernel"].append(rec)
        print(json.dumps(rec), flush=True)
    for n_snps, n_loci, reps, seed in ((150, 40, a.reps or 30, 7000), (1500, 4, a.reps or 3, 8000)):
        rec = batch_times(n_snps, n_loci, reps, seed)
        out["batch"].append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
