"""Cost of a grid of priors over a list of loci (pipsort_posterior_exhaustive_grid_batch), ms per locus, at c = 3:
  * 40 headline loci (150 SNPs per study, overlap 0.8, distinct seeds) and 4 loci of 1500 SNPs per study;
  * arms: the ordinary batch; the grid batch at 1 / 8 / 64 priors, full read and evidence read (every per-SNP member
    NULL); and, for the same 1 / 8 / 64 priors, as many ordinary batches (each with the loci carrying one prior) --
    what a grid costs without the class-resolved store.
Every call is synchronous (the host clock around it ends after the last read-back); the arms are interleaved within each
repetition, each warmed up first, and the median over the repetitions is reported.  The loci stay resident in L2 between
calls, as in bench.py's e2e arm.  The card's name and power limit are read in the same run.
python scripts/grid_batch_bench.py [--reps N] [--out file.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pipsort_b200 as P  # noqa: E402
from pipsort_b200 import synth  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0]


def priors(n):
    """n priors (gamma, p): 8 gammas from 1e-3 to 0.2 x n / 8 values of p in [0, 1]; one prior = the locus's own."""
    if n == 1:
        return [(0.01, 0.75)]
    g = np.geomspace(1e-3, 0.2, 8)
    p = np.linspace(0.0, 1.0, n // 8)
    return [(float(a), float(b)) for a in g for b in p]


def as_dict(L, **over):
    D = dict(num_snps=L.num_snps, sigma=np.concatenate([s.ravel() for s in L.sigma]), z=np.concatenate(L.z), d=L.d, K=L.K,
             snp_map=L.snp_map, gamma=L.gamma, sharing_param=L.sharing_param)
    D.update(over)
    return D


def measure(n_snps, n_loci, reps, seed):
    loci = [as_dict(synth.make_locus(n_snps, seed=seed + i)) for i in range(n_loci)]
    arms = {"ordinary": [P.LocusBatch(loci, 3)]}
    for k in (1, 8, 64):
        pr = priors(k)
        arms[f"grid_{k}"] = [P.LocusBatch(loci, 3, priors=pr)]
        arms[f"grid_{k}_evidence"] = [P.LocusBatch(loci, 3, priors=pr, evidence_only=True)]
        arms[f"ordinary_x{k}"] = [P.LocusBatch([dict(D, gamma=g, sharing_param=p) for D in loci], 3) for g, p in pr]
    for bs in arms.values():            # warm-up: modules, plans, the stream kits and staging of the engines in flight
        for _ in range(2):
            for b in bs:
                b.run()
    t = {name: [] for name in arms}
    for _ in range(reps):
        for name, bs in arms.items():
            t0 = time.perf_counter()
            for b in bs:
                b.run()
            t[name].append(1e3 * (time.perf_counter() - t0) / n_loci)
    # the evidence read gives the full read's scalars (1e-12: separate passes, atomics in another order)
    for k in (1, 8, 64):
        np.testing.assert_allclose(arms[f"grid_{k}_evidence"][0].evidence(), arms[f"grid_{k}"][0].evidence(), rtol=1e-12, atol=0)
    return {"snps_per_study": n_snps, "loci": n_loci, "reps": reps,
            "ms_per_locus": {name: float(np.median(v)) for name, v in t.items()},
            "ms_per_locus_min": {name: float(np.min(v)) for name, v in t.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=0, help="repetitions (default 30 for the 150-SNP list, 3 for the 1500-SNP one)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"gpu": gpu_info(), "c": 3, "runs": []}
    print(json.dumps({"gpu": out["gpu"]}), flush=True)
    for n_snps, n_loci, reps, seed in ((150, 40, a.reps or 30, 7000), (1500, 4, a.reps or 3, 8000)):
        rec = measure(n_snps, n_loci, reps, seed)
        out["runs"].append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
