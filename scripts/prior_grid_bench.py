"""Cost of a grid of priors (PIPSORT_PRIOR_CLASSES): on the 150- and 1500-SNP synthetic loci at c = 3, with the L2 flushed
before every launch, an ordinary engine and a class-resolved one interleaved step by step, it times
  * the exhaustive kernel of the ordinary pass and of the class-resolved pass (CUDA events around the kernel);
  * the read of the ordinary engine (finalize + copy back) and the grid read for 1, 8 and 64 priors (host clock around the
    synchronous call: prior upload, finalize over all priors, copy back, scatter);
and the number of priors above which one class-resolved pass + one grid read beats separate ordinary passes + reads.
python scripts/prior_grid_bench.py [--reps N] [--out file.json]"""
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
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().split("\n")[0]
    except OSError:
        return "unknown"


def priors(n):
    g = np.geomspace(1e-3, 0.2, 8)
    p = np.linspace(0.0, 1.0, max(n // 8, 1))
    return [(float(a), float(b)) for a in g for b in p][:n] if n >= 8 else [(0.01, 0.75)] * n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=0, help="timed repetitions (default 40 at 150 SNPs, 5 at 1500)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = {"gpu": gpu_info(), "c": 3, "loci": {}}
    for n, reps in ((150, a.reps or 40), (1500, a.reps or 5)):
        L = synth.make_locus(n)
        mk = lambda cr: P.Engine(L.num_snps, L.sigma, L.z, L.d, L.K, L.snp_map, gamma=L.gamma,  # noqa: E731
                                 sharing_param=L.sharing_param, max_causal=3, prior_classes=cr)
        eo, ec = mk(False), mk(True)
        for e in (eo, ec):                       # warm-up: modules, pair tables, plans
            for _ in range(3):
                e.reset(); e.run_exhaustive(3); e.read()
        grids = {k: priors(k) for k in (1, 8, 64)}
        for k, pr in grids.items():
            ec.read_prior_grid(pr)
        ko, kc, ro = [], [], []
        rg = {k: [] for k in grids}
        for _ in range(reps):
            eo.reset(); eo.flush_l2(); eo.run_exhaustive(3); ko.append(eo.last_kernel_ms())
            ec.reset(); ec.flush_l2(); ec.run_exhaustive(3); kc.append(ec.last_kernel_ms())
            eo.sync(); ec.sync()
            t0 = time.perf_counter(); eo.read(); ro.append(1e3 * (time.perf_counter() - t0))
            for k, pr in grids.items():
                t0 = time.perf_counter(); ec.read_prior_grid(pr); rg[k].append(1e3 * (time.perf_counter() - t0))
        med = lambda v: float(np.median(v))      # noqa: E731
        pass_o, pass_c, read_o = med(ko), med(kc), med(ro)
        rec = {"U": int(L.snp_map.shape[1]), "reps": reps, "kernel_ms_ordinary": pass_o, "kernel_ms_classes": pass_c,
               "ratio": pass_c / pass_o, "read_ms_ordinary": read_o,
               "grid_read_ms": {str(k): med(v) for k, v in rg.items()}}
        # n priors: n ordinary passes + reads against one class-resolved pass + one grid read (grid read cost interpolated
        # linearly between the measured sizes)
        xs, ys = [1, 8, 64], [rec["grid_read_ms"][str(k)] for k in (1, 8, 64)]
        be = None
        for m in range(1, 1025):
            if pass_c + float(np.interp(m, xs, ys, right=ys[-1] + (m - 64) * (ys[-1] - ys[1]) / 56)) < m * (pass_o + read_o):
                be = m
                break
        rec["break_even_priors"] = be
        out["loci"][str(n)] = rec
        print(json.dumps({str(n): rec}), flush=True)
        eo.close(); ec.close()
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
