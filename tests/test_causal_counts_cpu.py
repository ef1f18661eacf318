"""pipsort_count_posterior (count_posterior) and class_tables_from_counts on count tables: host code, the library is built, no
device is used.

The posterior and the log evidence are checked against a NumPy computation written here from the reference's log_prior
(postcal.cpp:19-59) on random tables, including its two special priors (p == 0 skips the sharing term, p == 1 gives a class
with a < J the weight 0) and -inf classes; class_tables_from_counts against a log-sum-exp over b0; every argument refusal.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.special import logsumexp

PIPSORT_E_ARG = 1


def ncnt(c):
    return (c + 1) * (c + 2) * (c + 3) // 6


def classes(c):
    return [(J, a, b0, J - a - b0) for J in range(c + 1) for a in range(J + 1) for b0 in range(J - a + 1)]


def log_w(c, g, p):
    """log pi'(J, a) of every count class (postcal.cpp:19-59 without U log(1-gamma))."""
    out = []
    for J, a, _, _ in classes(c):
        v = J * (np.log(g) - np.log1p(-g))
        if p == 1.0:
            v = v if a == J else -np.inf
        elif p != 0.0:
            v += a * np.log(p) + (J - a) * np.log((1 - p) / 2)
        out.append(v)
    return np.array(out)


def reference(tab, U, g, p):
    c = next(k for k in range(9) if ncnt(k) == tab.shape[1])
    lw = log_w(c, g, p)
    post = np.zeros((tab.shape[0], c + 1, c + 1, c + 1))
    ev = np.empty(tab.shape[0])
    for i in range(tab.shape[0]):
        x = lw + tab[i]
        tot = logsumexp(x)
        ev[i] = U[i] * np.log1p(-g) + tot
        for k, (J, a, b0, b1) in enumerate(classes(c)):
            post[i, a, b0, b1] = np.exp(x[k] - tot)
    return post, ev


def random_tables(n, c, seed, holes=0.1):
    rng = np.random.default_rng(seed)
    tab = rng.normal(-30.0, 15.0, size=(n, ncnt(c)))
    tab[:, 0] = rng.normal(-40.0, 5.0, size=n)            # J = 0: the null configuration is never empty
    tab[rng.random(tab.shape) < holes] = -np.inf
    tab[:, 0] = np.where(np.isneginf(tab[:, 0]), -40.0, tab[:, 0])
    return tab, rng.integers(1, 3000, size=n).astype(np.int32)


# ---- 1. against NumPy -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [0, 1, 2, 3, 5, 8])
@pytest.mark.parametrize("g,p", [(0.01, 0.75), (1e-3, 0.0), (0.2, 1.0), (0.01, 1e-9), (1e-6, 0.999999), (0.5, 0.25)])
def test_posterior_equals_numpy(c, g, p):
    import pipsort_b200 as P
    tab, U = random_tables(12, c, seed=c * 100 + int(g * 1e6) % 97)
    post, ev = P.count_posterior(tab, U, g, p)
    want, wev = reference(tab, U, g, p)
    assert post.shape == (12, c + 1, c + 1, c + 1)
    np.testing.assert_allclose(post, want, rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(ev, wev, rtol=1e-13, atol=0)
    np.testing.assert_allclose(post.sum(axis=(1, 2, 3)), 1.0, rtol=1e-13)
    A, B0, B1 = np.meshgrid(*[np.arange(c + 1)] * 3, indexing="ij")
    assert (post[:, A + B0 + B1 > c] == 0.0).all()


def test_special_priors():
    """p == 1: only a == J classes carry mass; p == 0: the sharing term is skipped (not the limit p -> 0)."""
    import pipsort_b200 as P
    tab, U = random_tables(5, 3, seed=7, holes=0.0)
    post, _ = P.count_posterior(tab, U, 0.01, 1.0)
    A, B0, B1 = np.meshgrid(*[np.arange(4)] * 3, indexing="ij")
    assert (post[:, (B0 + B1) > 0] == 0.0).all() and (post[:, B0 + B1 == 0] > 0.0).all()
    p0, _ = P.count_posterior(tab, U, 0.01, 0.0)
    tiny, _ = P.count_posterior(tab, U, 0.01, 1e-12)
    assert not np.allclose(p0, tiny)
    assert np.allclose(p0, reference(tab, U, 0.01, 0.0)[0], rtol=1e-12, atol=1e-300)


def test_marginals_and_evidence_agree_with_the_class_table_fit():
    """log_evidence is fit_prior's total at the same prior, on the class tables class_tables_from_counts makes."""
    import pipsort_b200 as P
    tab, U = random_tables(6, 3, seed=11)
    for g, p in ((0.01, 0.75), (1e-3, 0.0), (0.2, 1.0)):
        _, ev = P.count_posterior(tab, U, g, p)
        per = P.fit_prior(P.class_tables_from_counts(tab, 3), U, fit=0, gamma=g, p=p)[3]
        np.testing.assert_allclose(ev, per, rtol=1e-12, atol=0)


# ---- 2. class_tables_from_counts ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [0, 1, 3, 8])
def test_class_tables_from_counts(c):
    import pipsort_b200 as P
    tab, _ = random_tables(4, c, seed=40 + c, holes=0.3)
    tab[1, 1:] = -np.inf                                   # every class of J >= 1 empty
    got = P.class_tables_from_counts(tab, c)
    assert got.shape == (4, (c + 1) * (c + 2) // 2)
    for i in range(4):
        for J in range(c + 1):
            for a in range(J + 1):
                ks = [k for k, (JJ, aa, _, _) in enumerate(classes(c)) if JJ == J and aa == a]
                want = logsumexp(tab[i, ks]) if np.isfinite(tab[i, ks]).any() else -np.inf
                v = got[i, J * (J + 1) // 2 + a]
                assert (np.isneginf(v) and np.isneginf(want)) or v == pytest.approx(want, rel=1e-14, abs=1e-12)
    np.testing.assert_array_equal(P.class_tables_from_counts(tab[2]), got[2])
    with pytest.raises(ValueError):
        P.class_tables_from_counts(tab, c + 1)


# ---- 3. refusals ----------------------------------------------------------------------------------------------------------
def call(n_loci=2, c=1, tab=None, U=(5, 5), gamma=0.01, p=0.5):
    import pipsort_b200 as P
    from pipsort_b200.engine import _dp
    tab = np.zeros((2, ncnt(max(c, 0)))) if tab is None else tab
    Ua = np.ascontiguousarray(U, dtype=np.int32)
    post = np.empty(max(2 * ncnt(max(min(c, 8), 0)), 1))
    rc = P.lib().pipsort_count_posterior(n_loci, c, _dp(np.ascontiguousarray(tab, dtype=np.float64)),
                                         Ua.ctypes.data_as(C.POINTER(C.c_int32)), gamma, p, _dp(post), None)
    return rc, P.lib().pipsort_last_error().decode()


def table_with(i, k, v):
    t = np.zeros((2, 4))
    t[i, k] = v
    return t


@pytest.mark.parametrize("kw,text", [(dict(n_loci=0), "n_loci=0"), (dict(n_loci=-2), "n_loci=-2"), (dict(c=9), "c=9"),
                                     (dict(c=-1), "c=-1"), (dict(gamma=0.0), "gamma=0"), (dict(gamma=1.0), "gamma=1"),
                                     (dict(gamma=float("nan")), "gamma=nan"), (dict(p=-0.1), "sharing_param=-0.1"),
                                     (dict(p=1.5), "sharing_param=1.5"), (dict(p=float("nan")), "sharing_param=nan"),
                                     (dict(U=(5, 0)), "union_count[1]=0"), (dict(U=(-3, 5)), "union_count[0]=-3"),
                                     (dict(tab=table_with(1, 2, np.nan)), "tables[1][2]=nan"),
                                     (dict(tab=table_with(0, 3, np.inf)), "tables[0][3]=inf")])
def test_refusals_name_the_value(kw, text):
    rc, msg = call(**kw)
    assert rc == PIPSORT_E_ARG
    assert text in msg, msg


def test_locus_without_weighted_class_is_named():
    import pipsort_b200 as P
    tab = np.full((3, ncnt(1)), -np.inf)
    tab[:, 1] = 2.0                                        # (J = 1, a = 0, b0 = 0): zero weight at p = 1
    tab[[0, 2], 0] = -5.0
    with pytest.raises(P.PipsortError) as ei:
        P.count_posterior(tab, [4, 4, 4], 0.01, 1.0)
    assert ei.value.code == PIPSORT_E_ARG and "locus 1" in str(ei.value)
    post, _ = P.count_posterior(tab, [4, 4, 4], 0.01, 0.5)
    assert post[1, 0, 0, 1] == pytest.approx(1.0)


def test_python_refusals():
    import pipsort_b200 as P
    with pytest.raises(ValueError):
        P.count_posterior(np.zeros((2, 5)), [1, 1], 0.01, 0.5)      # 5 is no C(c+3, 3)
    with pytest.raises(ValueError):
        P.count_posterior(np.zeros((2, 4)), [1], 0.01, 0.5)
    with pytest.raises(ValueError):
        P.class_tables_from_counts(np.zeros((2, 5)))
    with pytest.raises(ValueError):
        P.LocusBatch([], 3, priors=[(0.01, 0.5)], count_table=True)
    with pytest.raises(ValueError):
        P.LocusBatch([], 3, class_evidence=True, count_table=True)
    assert P.count_table_batch([], 3).shape == (0, 20)
    with pytest.raises(P.PipsortError) as ei:
        P.count_table_batch([], 9)
    assert ei.value.code == PIPSORT_E_ARG and "c=9" in str(ei.value)
