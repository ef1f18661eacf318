"""CPU oracle of the count table (test infrastructure): R[a][b0][b1] of a locus, summed in log space over every expanded
configuration in the exhaustive walk's order -- union subsets of size J = 0..c, each SNP in every state its studies allow
(study 0 only, study 1 only, both).  Each configuration's likelihood is -K/2 + f_0(C0) + f_1(C1) with the oracle's f_block,
unweighted, the null configuration -K/2 - 1 (postcal.cpp:797-803).  Entry cnt_idx(J, a, b0) of the result is
logsumexp over the class, -inf for an empty class -- the layout of Engine.read_count_table."""
import itertools

import numpy as np
from scipy.special import logsumexp


def cnt_classes(c):
    """(J, a, b0, b1) of every entry of a count table up to c, in table order."""
    return [(J, a, b0, J - a - b0) for J in range(c + 1) for a in range(J + 1) for b0 in range(J - a + 1)]


def count_table(L, c):
    """L: oracle Locus (or anything with n_snps / num_snps, sigma, z, d, K, snp_map).  Returns (table, n_configs)."""
    from oracle import oracle as O
    smap = np.asarray(L.snp_map)
    U = smap.shape[1]
    sig = [np.ascontiguousarray(s, dtype=np.float64) for s in L.sigma]
    z = [np.ascontiguousarray(v, dtype=np.float64) for v in L.z]
    d = [float(v) for v in L.d]
    cache = [{}, {}]

    def f(s, idx):
        key = tuple(sorted(idx))
        v = cache[s].get(key)
        if v is None:
            v = cache[s][key] = O.f_block(sig[s], z[s], d[s], list(key)) if key else 0.0
        return v

    index = {(J, a, b0): k for k, (J, a, b0, _) in enumerate(cnt_classes(c))}
    vals = [[] for _ in index]
    vals[0].append(-0.5 * L.K - 1.0)
    n = 1
    for J in range(1, min(c, U) + 1):
        for sub in itertools.combinations(range(U), J):
            opts = []
            for g in sub:
                h0, h1 = smap[0, g] >= 0, smap[1, g] >= 0
                opts.append([t for t, ok in ((0, h0), (1, h1), (2, h0 and h1)) if ok])
            for st in itertools.product(*opts):
                c0 = [int(smap[0, g]) for g, t in zip(sub, st) if t != 1]
                c1 = [int(smap[1, g]) for g, t in zip(sub, st) if t != 0]
                a, b0 = st.count(2), st.count(0)
                vals[index[(J, a, b0)]].append(-0.5 * L.K + f(0, c0) + f(1, c1))
                n += 1
    tab = np.array([logsumexp(v) if v else -np.inf for v in vals])
    return tab, n
