"""The loci of test_gpu_extended_range.py really leave the exhaustive kernel's fast range where they are meant to.

classify() restates the kernel's routing (exhaustive_dev.cuh: okA / okb / okX, the pair table's +inf entries, the high-word
check of E{a,b,x}) in float64; these tests keep the loci from quietly falling back into the fast range when synth or a seed
changes.  No GPU needed.
"""
import numpy as np
import pytest

import range_loci as R


@pytest.fixture(scope="module")
def straddle():
    return R.straddle_locus()


@pytest.fixture(scope="module")
def threshold():
    return R.threshold_locus()


def _name(k):
    return f"{R.KIND_NAMES[k[0]]} trigger in study {k[1]}, x of type {k[2]}"


@pytest.mark.parametrize("keep_order", [False, True])
def test_straddle_locus_covers_every_trigger(straddle, keep_order):
    """Every trigger x study x type of x has a slow subset in a warp-step that also has fast lanes, for pairs and triples,
    in the engine's order and in the snp_map order."""
    cl = R.classify(straddle, keep_order)
    for J in (2, 3):
        missing = R.required_coverage(J) - cl[J].coverage()
        assert not missing, f"J={J}: " + "; ".join(_name(k) for k in sorted(missing))
        # most subsets stay fast: the slow path is exercised next to the fast one, not instead of it
        assert 0.05 < cl[J].slow.mean() < 0.6


def test_straddle_locus_strengths(straddle):
    """Per study: single SNPs in (2^440, 2^450) and above 2^450, pairs beyond 2^450 of fast singles, triples beyond 2^450
    of fast pairs; nothing beyond what the exponent store holds comfortably."""
    cl = R.classify(straddle)
    for s in range(2):
        n = len(straddle.z[s])
        single = R.log2_e(straddle, s, np.arange(n)[:, None])
        slow1 = R.e1n(straddle, s) >= R.E1_LIMIT
        assert ((single > 440) & (single < 450) & slow1).sum() >= 2
        assert ((single > 450) & slow1).sum() >= 2
        assert single.max() < 460
        assert (cl[2].trig[:, s] == R.PAIR).sum() >= 5
        assert (cl[3].trig[:, s] == R.TRIPLE).sum() >= 20


def test_straddle_locus_results_are_negative_and_moderate(straddle):
    """K puts every log-space result of the class-3 run below 0 and within a few thousand nats (relative tolerances mean
    something, and no result is the 0.0 that stands for "empty")."""
    from conftest import synth_as_oracle_locus
    from oracle import oracle as O
    r = O.exhaustive(synth_as_oracle_locus(straddle), 3)
    vals = np.concatenate([[r.total], r.post, r.noCausal, r.sharedPips[r.sharedPips != 0], r.sharedLL[r.sharedLL != 0],
                           r.notSharedLL])
    assert np.all(vals < -50.0) and np.all(vals > -5000.0)
    assert np.all(r.post != 0) and np.all(r.notSharedLL != 0)


def _case_row(L, cl, where, name):
    perm = R.order(L.snp_map)
    pos = sorted(np.argsort(perm)[where[name]])
    r = cl[len(pos)]
    return r, int(np.nonzero((r.idx == pos).all(1))[0][0])


def test_threshold_locus_sits_on_the_limits(threshold):
    L, where = threshold
    cl = R.classify(L)
    for name, s, kind, snps, target in R.THRESHOLD_CASES:
        if kind == R.SINGLE:
            i = int(L.snp_map[s, where[name][0]])
            A = 1.0 + L.d[s] * L.sigma[s][i, i]
            v = 0.5 * L.d[s] * L.z[s][i] ** 2 / A * R.LOG2E
            assert v == pytest.approx(target, abs=1e-9)
            if name.endswith("below"):
                assert R.e1n(L, s)[i] == R.E1_LIMIT - 1
            elif name.endswith("above"):
                assert R.e1n(L, s)[i] == R.E1_LIMIT
            else:
                assert abs(v / (R.E1_LIMIT - 0.5) - 1.0) <= 1e-12
            # paired with a SNP the study lacks, the SNP is the study's whole subset: below the limit the study's part stays
            # fast, above it the single SNP sends the pair down the slow path
            perm = R.order(L.snp_map)
            p = int(np.argsort(perm)[where[name][0]])
            rows = [r for r in np.nonzero((cl[2].idx == p).any(1))[0]
                    if all(L.snp_map[s, perm[u]] < 0 for u in cl[2].idx[r] if u != p)]
            assert rows
            want = {"below": R.FAST, "above": R.SINGLE}.get(name.split("_")[1])
            if want is not None:
                assert all(cl[2].trig[r, s] == want for r in rows)
            continue
        r, row = _case_row(L, cl, where, name)
        v = r.log2e[row, s]
        assert v == pytest.approx(target, abs=1e-9)
        if name.endswith("near"):
            assert abs(2.0 ** (v - R.FAST_BITS) - 1.0) <= 1e-12
        # the case's only reason to leave the fast range is the value at the limit
        other = 1 - s
        assert r.trig[row, other] == R.FAST
        if name.endswith("below"):
            assert r.trig[row, s] == R.FAST
        elif name.endswith("above"):
            assert r.trig[row, s] == kind
            assert r.mixed_steps()[row]
        else:
            assert r.trig[row, s] in (R.FAST, kind)
