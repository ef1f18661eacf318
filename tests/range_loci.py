"""Loci that leave the exhaustive kernel's fast range, and the kernel's routing predicate restated in float64 numpy.

The register kernel (pipsort_b200/csrc/exhaustive_dev.cuh) evaluates a pair or triple with plain doubles only while every
E_s(C) = exp(f_s(C)) it touches stays below 2^450; otherwise the subset goes down the mantissa/exponent path (slow_subset).
Per study s the subset is sent there by
  single  a member SNP whose rounded exponent of exp(d/2 z^2 / A) is >= 440 (`e1n`, the okA / okb / okX checks);
  pair    two members with E{i,j} >= 2^450 (the pair table's +inf entries: v3, v5 and e6 in the step);
  triple  all three members in the study and E{a,b,x} >= 2^450 (the high-word check of e7).
The loci here are built from pipsort_b200.synth with a few z-scores solved from the closed forms, so that every trigger
occurs in both studies, next to fast subsets of the same warp-step, for every type of x.

Test infrastructure only (numpy + scipy); f_s(C) = d/2 z_C' M^-1 z_C - 1/2 log det M with M = I + d Sigma_C.
"""
from __future__ import annotations

import dataclasses
import itertools

import numpy as np

from pipsort_b200 import synth

LN2 = float(np.log(2.0))
LOG2E = 1.4426950408889634
E1_LIMIT = 440          # single-SNP switch: xexp exponent of exp(d/2 z^2/A) (rounded to nearest) >= 440
FAST_BITS = 450.0       # E >= 2^450 leaves the fast range
FAST, SINGLE, PAIR, TRIPLE = 0, 1, 2, 3
KIND_NAMES = {SINGLE: "single", PAIR: "pair", TRIPLE: "triple"}


# ---- f_s(C) in float64 ----------------------------------------------------------------------------------------------
def log_e(L, s, idx):
    """f_s(C) in nats for study-local index sets idx [..., k] (every index present in study s)."""
    idx = np.asarray(idx, dtype=np.int64)
    sig, z, d = np.asarray(L.sigma[s]), np.asarray(L.z[s]), float(L.d[s])
    k = idx.shape[-1]
    M = np.eye(k) + d * sig[idx[..., :, None], idx[..., None, :]]
    zc = z[idx]
    sol = np.linalg.solve(M, zc[..., None])[..., 0]
    _, ld = np.linalg.slogdet(M)
    return 0.5 * d * (zc * sol).sum(-1) - 0.5 * ld


def log2_e(L, s, idx):
    return log_e(L, s, idx) / LN2


def e1n(L, s):
    """The kernel's exponent of E_s({i}) per study-local SNP: rint(d/2 z^2/A * log2 e)."""
    sig, z, d = np.asarray(L.sigma[s]), np.asarray(L.z[s]), float(L.d[s])
    A = 1.0 + d * np.diag(sig)
    return np.rint(0.5 * d * (z * z / A) * LOG2E).astype(np.int64)


def _types(smap):
    return np.where((smap[0] >= 0) & (smap[1] >= 0), 0, np.where(smap[0] >= 0, 1, np.where(smap[1] >= 0, 2, 3)))


def _tiles(types):
    """Tile of every x (exh_plan.h ExhTiles): 32-wide tiles that end at the boundaries between SNP types."""
    U = len(types)
    cut = [0] + [i for i in range(1, U) if types[i] != types[i - 1]]
    if len(cut) > 4:
        cut = [0]
    cut.append(U)
    of, T = np.zeros(U, dtype=np.int64), 0
    for g0, g1 in zip(cut, cut[1:]):
        nt = (g1 - g0 + 31) // 32
        for j in range(nt):
            lo = g1 - 32 * (nt - j)
            of[max(lo, g0):lo + 32] = T
            T += 1
    return of


@dataclasses.dataclass
class Routing:
    """classify() for one size class: subsets in the kernel's working order (rows of `idx`, internal union positions)."""
    idx: np.ndarray        # [n, J] internal positions, increasing
    trig: np.ndarray       # [n, 2] per study: FAST / SINGLE / PAIR / TRIPLE (the first trigger that applies, in that order)
    xtype: np.ndarray      # [n] type of x (the last SNP): 0 both studies, 1 study 0 only, 2 study 1 only
    step: np.ndarray       # [n] id of the warp-step (a, b, tile of x): lanes of one step run together
    log2e: np.ndarray      # [n, 2] log2 E_s(subset) (nan where the study has none of its SNPs)

    @property
    def slow(self):
        return (self.trig != FAST).any(1)

    def mixed_steps(self):
        """Mask of the subsets whose warp-step has fast and slow lanes."""
        sl = self.slow
        has_slow = np.zeros(self.step.max() + 1, bool)
        has_fast = np.zeros_like(has_slow)
        has_slow[self.step[sl]] = True
        has_fast[self.step[~sl]] = True
        return has_slow[self.step] & has_fast[self.step]

    def coverage(self):
        """{(kind, study, type of x)} of the slow subsets that share their warp-step with fast ones."""
        m = self.mixed_steps()
        out = set()
        for s in range(2):
            for k in (SINGLE, PAIR, TRIPLE):
                for t in np.unique(self.xtype[m & (self.trig[:, s] == k)]):
                    out.add((k, s, int(t)))
        return out


def order(smap, keep_order=False):
    """Internal order of the engine (union SNPs stably sorted by type) or the snp_map order: perm[i] = union index."""
    t = _types(smap)
    return np.arange(len(t)) if keep_order else np.argsort(t, kind="stable")


def classify(L, keep_order=False):
    """{2: Routing of the pairs, 3: Routing of the triples} as the kernel routes them (engine order by default)."""
    smap = np.asarray(L.snp_map)
    perm = order(smap, keep_order)
    U = len(perm)
    loc = smap[:, perm]                       # [2, U] study-local index per internal position, -1 when absent
    types = _types(loc)
    tile = _tiles(types)
    slow1 = np.zeros((2, U), bool)
    pair_bits = np.full((2, U, U), np.nan)
    for s in range(2):
        pres = np.nonzero(loc[s] >= 0)[0]
        slow1[s, pres] = e1n(L, s)[loc[s, pres]] >= E1_LIMIT
        ij = np.array([(i, j) for i in pres for j in pres if i < j], dtype=np.int64).reshape(-1, 2)
        if len(ij):
            v = log2_e(L, s, loc[s][ij])
            pair_bits[s, ij[:, 0], ij[:, 1]] = v
            pair_bits[s, ij[:, 1], ij[:, 0]] = v
    out = {}
    for J in (2, 3):
        idx = np.array(list(itertools.combinations(range(U), J)), dtype=np.int64).reshape(-1, J)
        n = len(idx)
        trig = np.zeros((n, 2), dtype=np.int64)
        bits = np.full((n, 2), np.nan)
        for s in range(2):
            pr = loc[s][idx] >= 0                                          # [n, J]
            single = (pr & slow1[s][idx]).any(1)
            pair = np.zeros(n, bool)
            for u, w in itertools.combinations(range(J), 2):
                pb = pair_bits[s, idx[:, u], idx[:, w]]
                pair |= pr[:, u] & pr[:, w] & (pb >= FAST_BITS)
            anyp = pr.any(1)
            if anyp.any():
                sub = np.nonzero(anyp)[0]
                # f of the study's part of the subset (absent SNPs are virtual: they leave E unchanged)
                for k in range(1, J + 1):
                    rows = sub[pr[sub].sum(1) == k]
                    if len(rows):
                        li = np.array([loc[s][idx[r]][pr[r]] for r in rows], dtype=np.int64)
                        bits[rows, s] = log2_e(L, s, li)
            full = pr.all(1) & (bits[:, s] >= FAST_BITS) if J == 3 else np.zeros(n, bool)
            trig[:, s] = np.where(single, SINGLE, np.where(pair, PAIR, np.where(full, TRIPLE, FAST)))
        xtype = types[idx[:, -1]]
        key = (idx[:, -3] * U if J == 3 else 0) * U + idx[:, -2] * U + tile[idx[:, -1]]
        _, step = np.unique(key, return_inverse=True)
        out[J] = Routing(idx, trig, xtype, step.ravel(), bits)
    return out


def required_coverage(J):
    """Every (trigger, study, type of x) that can occur in a warp-step with fast lanes.  A trigger on a or b makes the whole
    step slow, so in a mixed step the trigger involves x, and x is in the trigger's study (not of the other study only)."""
    return {(k, s, t) for s in range(2) for k in (SINGLE, PAIR) + ((TRIPLE,) if J == 3 else ()) for t in (0, 1 + s)}


# ---- builders -------------------------------------------------------------------------------------------------------
def z_for_bits(L, s, i, bits, sign=1.0):
    """z of study-local SNP i such that log2 E_s({i}) = bits:  f = d/2 z^2/A - 1/2 log A."""
    d = float(L.d[s])
    A = 1.0 + d * float(L.sigma[s][i, i])
    return sign * np.sqrt((bits * LN2 + 0.5 * np.log(A)) * A / (0.5 * d))


def choose_K(L, c=5, margin_nats=200.0):
    """K (= S'S, a free input) such that every log-space result is negative and a few thousand nats at most: the shift
    -K/2 lies above the largest contribution of up to c causal SNPs, bounded per study by the largest f of at most three
    SNPs (z-scores set by hand need not fit the LD, so pairs and triples can exceed their singles by far) plus the c - 3
    largest singles, plus a margin."""
    top = 0.0
    for s in range(2):
        n = len(L.z[s])
        f1 = log_e(L, s, np.arange(n)[:, None])
        best = float(max(f1.max(initial=0.0), 0.0))
        for k in (2, 3):
            if n >= k:
                best = max(best, float(log_e(L, s, np.array(list(itertools.combinations(range(n), k)))).max()))
        top += best + float(np.sort(np.maximum(f1, 0.0))[::-1][:max(c - 3, 0)].sum())
    return 2.0 * (top + margin_nats)


def _with_z(L, z, K=None):
    L = dataclasses.replace(L, z=[np.array(v, dtype=np.float64) for v in z])
    return dataclasses.replace(L, K=choose_K(L) if K is None else K)


def _groups(smap):
    """Union positions (snp_map order) of the shared SNPs and of each study's own SNPs."""
    t = _types(smap)
    return np.nonzero(t == 0)[0], np.nonzero(t == 1)[0], np.nonzero(t == 2)[0]


# per study: which SNP of which type group gets which strength (log2 E{i}); groups (shared, the study's own), position
# in the group.  Strong single SNPs at the first and last position of every group (in the roles a, b and x), a few SNPs
# whose pairs leave the fast range, and more whose pairs stay in it but whose triples do not; different SNPs per study.
STRADDLE_PLAN = {
    0: [("sh", 0, 445.0), ("sh", -1, 455.0), ("own", 0, 455.0), ("own", -1, 445.0),
        ("sh", 2, 300.0), ("sh", -3, 300.0), ("own", 2, 300.0),
        ("sh", 1, 200.0), ("sh", -2, 200.0), ("sh", 4, 200.0), ("own", 1, 200.0), ("own", -2, 200.0)],
    1: [("sh", 0, 455.0), ("sh", -1, 445.0), ("own", 0, 445.0), ("own", -1, 455.0),
        ("sh", 3, 300.0), ("sh", -4, 300.0), ("own", 3, 300.0),
        ("sh", 5, 200.0), ("sh", -5, 200.0), ("sh", 6, 200.0), ("own", 1, 200.0), ("own", -2, 200.0)],
}


def straddle_locus(n_per_study=40, overlap=0.5, seed=77, sharing_param=0.75):
    """make_locus(40, overlap=0.5) (U = 60, 20 SNPs of each type) with the z of 12 SNPs per study overwritten so that every
    trigger of the slow path occurs in both studies, at the first and last positions of the type groups (the roles a, b
    and x in both SNP orders)."""
    SL = synth.make_locus(n_per_study, overlap=overlap, seed=seed, sharing_param=sharing_param)
    smap = SL.snp_map
    sh, o0, o1 = _groups(smap)
    z = [np.array(v) for v in SL.z]
    for s in range(2):
        own = (o0, o1)[s]
        for grp, pos, bits in STRADDLE_PLAN[s]:
            g = (sh if grp == "sh" else own)[pos]
            i = int(smap[s, g])
            z[s][i] = z_for_bits(SL, s, i, bits, 1.0 if z[s][i] >= 0 else -1.0)
    return _with_z(SL, z)


def lone_strong_locus(n_per_study=40, overlap=0.5, seed=77, bits=455.0):
    """The base locus of straddle_locus with ONE strong SNP: the first study-0-only SNP at 2^bits in study 0, all else weak.
    Then the subsets that hold it dominate the accumulators they touch, also those whose other SNPs are of study 1 only
    (a in study 0 alone, b and x in study 1 alone: the kernel must route them by the single trigger of a, not by b or x)."""
    SL = synth.make_locus(n_per_study, overlap=overlap, seed=seed)
    _, o0, _ = _groups(SL.snp_map)
    i = int(SL.snp_map[0, o0[0]])
    # the strong SNP outside every LD block: its z fits the LD, and a SNP next to it adds its own E, not a residual of it
    sig0 = np.array(SL.sigma[0])
    sig0[i, :] = 0.0
    sig0[:, i] = 0.0
    sig0[i, i] = 1.0
    SL = dataclasses.replace(SL, sigma=[sig0, SL.sigma[1]])
    z = [np.array(v) for v in SL.z]
    z[0][i] = z_for_bits(SL, 0, i, bits)
    return _with_z(SL, z)


def spread_locus(n_per_study=12, d0=1e12, seed=31):
    """All SNPs shared, study 0 with a huge d (a sample-size ratio of ~10^11) and tiny z: every causal SNP of study 0 lowers
    E_0 by ~20 bits (1/sqrt(A), A ~ d0), so within one configuration of k SNPs the expansions span ~20 k bits (2^-160 for
    8 SNPs) in the determinant factor, while the exponents of exp(d/2 q) stay put."""
    SL = synth.make_locus(n_per_study, overlap=1.0, seed=seed)
    # study-0 z of ~1e-5: d0/2 |z|^2 stays within the exponent range the engine provisions (create refuses more)
    SL = dataclasses.replace(SL, d=np.array([d0, float(SL.d[1])]), z=[1e-5 * np.asarray(SL.z[0]), 0.3 * np.asarray(SL.z[1])])
    return dataclasses.replace(SL, K=choose_K(SL, c=8))


def _solve_z(L, s, members, who, target_bits, z):
    """brentq on z[s][who] (who in members, study-local) so that log2 E_s(members) = target_bits.  f is a convex quadratic
    in z[s][who]: the root is taken on the increasing side of its minimum (where the SNP's residual vanishes)."""
    from scipy.optimize import brentq
    members = np.asarray(members, dtype=np.int64)
    k = int(np.nonzero(members == who)[0][0])
    Minv = np.linalg.inv(np.eye(len(members)) + float(L.d[s]) * np.asarray(L.sigma[s])[np.ix_(members, members)])
    zc = z[s][members].copy()
    zc[k] = 0.0
    zmin = -float(Minv[k] @ zc) / Minv[k, k]

    def g(v):
        zz = [np.array(q) for q in z]
        zz[s][who] = v
        return log2_e(dataclasses.replace(L, z=zz), s, members) - target_bits

    assert g(zmin) < 0.0, "the other SNPs of the case alone are beyond the target"
    step = 1.0
    while g(zmin + step) <= 0.0:
        step *= 2.0
    z[s][who] = brentq(g, zmin, zmin + step, xtol=1e-15, rtol=8.9e-16, maxiter=500)


# Boundary cases of threshold_locus: (name, study, kind, union SNPs as (group, position), target)
#   single: the kernel's exponent t log2 e (t = d/2 z^2/A) at the rounding boundary 439.5 of e1n, 0.01 bit off or within
#           1e-12 relative;  pair / triple: log2 E of the subset at 450 +- 0.01 bit, or E within 1e-12 relative of 2^450.
NEAR = 1e-12 / 3
THRESHOLD_CASES = [
    ("single_below", 0, SINGLE, [("own", 0)], E1_LIMIT - 0.5 - 0.01),
    ("single_above", 1, SINGLE, [("own", 0)], E1_LIMIT - 0.5 + 0.01),
    ("single_near", 0, SINGLE, [("sh", 0)], (E1_LIMIT - 0.5) * (1.0 - NEAR)),
    ("pair_below", 0, PAIR, [("sh", 1), ("own", 1)], FAST_BITS - 0.01),
    ("pair_above", 1, PAIR, [("sh", 2), ("own", 1)], FAST_BITS + 0.01),
    ("pair_near", 0, PAIR, [("own", 2), ("own", 3)], FAST_BITS + np.log2(1.0 + NEAR)),
    ("triple_below", 0, TRIPLE, [("sh", 3), ("own", 4), ("own", 5)], FAST_BITS - 0.01),
    ("triple_above", 1, TRIPLE, [("sh", 4), ("own", 2), ("own", 3)], FAST_BITS + 0.01),
    ("triple_near", 1, TRIPLE, [("sh", 5), ("own", 4), ("own", 5)], FAST_BITS + np.log2(1.0 - NEAR)),
]


def threshold_locus(seed=5, background=0.05, ld_scale=0.3, sharing_param=0.75):
    """make_locus(12, overlap=0.5) (U = 18, 6 SNPs of each type) with weak background z-scores and, per boundary case
    (THRESHOLD_CASES), the z of one SNP found by root finding so that the case's value sits right at a range limit.
    Returns (locus, {case name: sorted union positions of the case's SNPs})."""
    SL = synth.make_locus(12, overlap=0.5, seed=seed, sharing_param=sharing_param)
    # LD shrunk towards the identity (correlations <= ld_scale): the SNPs of one case stay apart from each other
    SL = dataclasses.replace(SL, sigma=[(1.0 - ld_scale) * np.eye(len(v)) + ld_scale * np.asarray(v) for v in SL.sigma])
    smap = SL.snp_map
    sh, o0, o1 = _groups(smap)
    z = [background * np.array(v) for v in SL.z]
    where = {}
    for name, s, kind, snps, target in THRESHOLD_CASES:
        own = (o0, o1)[s]
        g = [int((sh if grp == "sh" else own)[pos]) for grp, pos in snps]
        li = [int(smap[s, u]) for u in g]
        where[name] = sorted(g)
        if kind == SINGLE:
            d = float(SL.d[s])
            A = 1.0 + d * float(SL.sigma[s][li[0], li[0]])
            z[s][li[0]] = np.sqrt(target / LOG2E * A / (0.5 * d))
        else:
            for u in li[:-1]:                                   # the others: well inside the fast range (pairs < 2^450)
                z[s][u] = z_for_bits(SL, s, u, 450.0 / len(li) - 10.0 * (len(li) - 2) - 25.0)
            _solve_z(SL, s, li, li[-1], target, z)
    return _with_z(SL, z), where
