"""ms per locus of the shotgun search over a list of loci: one-at-a-time pipsort_sss (a fresh Engine per locus: create, search,
read, destroy) against pipsort_sss_batch at 1 .. 4 searches in flight per host thread (PIPSORT_SSS_DEPTH), on 1 and 3 host
threads (PIPSORT_BATCH_THREADS is read once per process: one child process per thread count).  Host clock around each
synchronous call; the modes alternate within every repetition and the median is reported.

Lists: (a) 40 distinct synthetic loci of 150 SNPs per study, c = 3; (b) 8 flat loci shaped like tests/search_loci.py
(16 SNPs per study, no causal SNP) at c = 6: nearly flat likelihoods, so the searches climb towards states of c SNPs and
run more rounds than on loci with strong SNPs; (c) 4 loci of 5000 SNPs per study, c = 5 (BASELINE.json configs[4]).

    python scripts/sss_batch_bench.py [--reps 5] [--lists a,b,c] [--out results.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEPTHS = (1, 2, 3, 4)


def make_list(name):
    """(loci as LocusBatch takes them, c)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import search_loci as S
    from pipsort_b200 import synth
    if name == "a":
        L, c = [synth.make_locus(150, overlap=0.8, seed=3000 + i) for i in range(40)], 3
    elif name == "b":
        L, c = [S.flat_locus(16, 0.6, seed, 0.3) for seed in range(3, 11)], 6
    else:
        L, c = [synth.make_locus(5000, overlap=0.8, seed=20261018 + i) for i in range(4)], 5
    D = [dict(num_snps=np.asarray(x.num_snps, dtype=np.int32), sigma=np.concatenate([np.ravel(s) for s in x.sigma]),
              z=np.concatenate(x.z), d=np.asarray(x.d, dtype=np.float64), K=float(x.K), snp_map=np.asarray(x.snp_map, dtype=np.int32),
              gamma=float(x.gamma), sharing_param=float(x.sharing_param)) for x in L]
    return D, c


def child(lists, reps):
    import pipsort_b200 as P
    out = {}
    for name in lists:
        D, c = make_list(name)

        def one_at_a_time():
            r = []
            for Lc in D:
                with P.Engine(Lc["num_snps"], Lc["sigma"], Lc["z"], Lc["d"], Lc["K"], Lc["snp_map"], gamma=Lc["gamma"],
                              sharing_param=Lc["sharing_param"], max_causal=c) as e:
                    r.append(e.sss(c)[1])
            return r

        B = P.LocusBatch(D, c, search=True)

        def batched(depth):
            os.environ["PIPSORT_SSS_DEPTH"] = str(depth)
            B.run()
            return B.iterations.tolist()

        modes = [("one_at_a_time", one_at_a_time)] + [(f"batch_depth{d}", lambda d=d: batched(d)) for d in DEPTHS]
        rounds = one_at_a_time()                                   # warm-up of every mode (streams, pools, plans)
        for _, f in modes:
            assert f() == rounds
        times = {m: [] for m, _ in modes}
        for _ in range(reps):
            for m, f in modes:
                t = time.perf_counter()
                f()
                times[m].append(1e3 * (time.perf_counter() - t) / len(D))
        out[name] = dict(c=c, n_loci=len(D), mean_rounds=sum(rounds) / len(rounds),
                         ms_per_locus={m: statistics.median(v) for m, v in times.items()},
                         spread={m: [min(v), max(v)] for m, v in times.items()})
    print("RESULT " + json.dumps(out), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lists", default="a,b,c")
    ap.add_argument("--out")
    ap.add_argument("--child", action="store_true")
    a = ap.parse_args()
    lists = a.lists.split(",")
    if a.child:
        sys.path.insert(0, ROOT)
        return child(lists, a.reps)
    gpu = card()
    print(f"card, power limit, max SM clock: {gpu}", flush=True)
    res = {}
    for T in (1, 3):
        env = dict(os.environ, PIPSORT_BATCH_THREADS=str(T))
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--reps", str(a.reps), "--lists", a.lists],
                           env=env, capture_output=True, text=True)
        if p.returncode != 0:
            sys.exit(f"child with {T} threads failed:\n{p.stderr[-3000:]}")
        res[T] = json.loads(next(x for x in p.stdout.splitlines() if x.startswith("RESULT "))[7:])
    print("| list | threads | mean rounds | one at a time | " + " | ".join(f"batch, depth {d}" for d in DEPTHS) + " |")
    print("|---|---|---|---|" + "---|" * len(DEPTHS))
    for name in lists:
        for T in (1, 3):
            r = res[T][name]
            ms = r["ms_per_locus"]
            print(f"| ({name}) {r['n_loci']} loci, c = {r['c']} | {T} | {r['mean_rounds']:.1f} | {ms['one_at_a_time']:.3f} | "
                  + " | ".join(f"{ms[f'batch_depth{d}']:.3f}" for d in DEPTHS) + " |")
    if a.out:
        with open(a.out, "w") as f:
            json.dump(dict(card=gpu, results=res), f, indent=1)


if __name__ == "__main__":
    main()
