"""Cost of choosing the prior by marginal likelihood, at c = 3:
  * ms per locus of the class-table batch (pipsort_class_evidence_batch) against the ordinary batch and the evidence-only
    grid batch at 64 priors (what a caller scanning a grid pays instead), on 40 loci of 150 SNPs per study (overlap 0.8,
    distinct seeds) and 4 loci of 1500 SNPs per study;
  * ms of pipsort_fit_prior alone (host code) on 10^4 synthetic class tables, fitting p and fitting (gamma, p).
Every call is synchronous (the host clock around it ends after the last read-back); the device arms are interleaved within
each repetition, each warmed up first, and the median over the repetitions is reported.  The loci stay resident in L2
between calls, as in bench.py's e2e arm and scripts/grid_batch_bench.py.  The card's name and power limit are read in the
same run.
python scripts/prior_fit_bench.py [--reps N] [--out file.json]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from grid_batch_bench import as_dict, gpu_info, priors  # noqa: E402
import pipsort_b200 as P  # noqa: E402
from pipsort_b200 import synth  # noqa: E402


def measure(n_snps, n_loci, reps, seed):
    loci = [as_dict(synth.make_locus(n_snps, seed=seed + i)) for i in range(n_loci)]
    arms = {"ordinary": P.LocusBatch(loci, 3),
            "grid_64_evidence": P.LocusBatch(loci, 3, priors=priors(64), evidence_only=True),
            "class_tables": P.LocusBatch(loci, 3, class_evidence=True)}
    for b in arms.values():             # warm-up: modules, plans, the stream kits and staging of the engines in flight
        for _ in range(2):
            b.run()
    t = {name: [] for name in arms}
    for _ in range(reps):
        for name, b in arms.items():
            t0 = time.perf_counter()
            b.run()
            t[name].append(1e3 * (time.perf_counter() - t0) / n_loci)
    # the tables give the evidence read's totals (1e-12: separate passes, atomics in another order)
    tabs, U = arms["class_tables"].tables(), [L["snp_map"].shape[1] for L in loci]
    ev = arms["grid_64_evidence"].evidence()[:, :, 0]
    for j, (g, p) in enumerate(priors(64)):
        np.testing.assert_allclose(P.fit_prior(tabs, U, fit=0, gamma=g, p=p)[3], ev[:, j], rtol=1e-12, atol=0)
    return {"snps_per_study": n_snps, "loci": n_loci, "reps": reps,
            "ms_per_locus": {name: float(np.median(v)) for name, v in t.items()},
            "ms_per_locus_min": {name: float(np.min(v)) for name, v in t.items()}}


def fit_times(n_tables, reps):
    """pipsort_fit_prior on n_tables class tables of c = 3 with the shape of real ones (T[0][0] = 1; classes J >= 1 from
    a shared and an ancestry-specific signal strength per locus)."""
    rng = np.random.default_rng(5)
    J = np.array([j for j in range(4) for _ in range(j + 1)])
    a = np.array([k for j in range(4) for k in range(j + 1)])
    sh, own = rng.uniform(0, 14, (n_tables, 1)), rng.uniform(0, 14, (n_tables, 1))
    scale = np.sqrt(np.maximum(J, 1)) / np.maximum(J, 1)
    tab = (a * sh + (J - a) * own) * scale + rng.normal(0, 0.3, (n_tables, 10)) * (J > 0) - rng.uniform(0, 3, (n_tables, 1))
    U = rng.integers(2, 30, n_tables)
    out = {"tables": n_tables, "reps": reps}
    for fit in ("p", "gamma,p"):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            r = P.fit_prior(tab, U, fit=fit)
            ts.append(1e3 * (time.perf_counter() - t0))
        out[fit] = {"ms": float(np.median(ts)), "gamma": r[0], "p": r[1]}
    return out


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
    out["fit"] = fit_times(10000, 3)
    print(json.dumps({"fit": out["fit"]}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
