"""pipsort_fit_prior (fit_prior): the joint log evidence of class tables and the prior that maximises it.  Host code: the
library is built, no device is used.

The evaluation (fit=0) is checked against a log-sum-exp written here from the reference's log_prior (postcal.cpp:19-59),
including its two special priors: p == 0 skips the sharing term, p == 1 gives a class with a < J the weight 0.  The fits are
checked against scipy (a dense grid, then minimize_scalar(method="bounded"), one coordinate at a time), and tables built for
one documented answer each: p = 0 (the skip rule) outweighing every p in (0, 1] and therefore never the fit of p, a p = 1
optimum, a bimodal objective whose global maximum lies in the narrower basin, and -inf classes.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.optimize import minimize_scalar
from scipy.special import logsumexp

PIPSORT_E_ARG = 1


def ntab(c):
    return (c + 1) * (c + 2) // 2


def log_pi(c, g, p):
    """log pi'(J, a) in class order J (J+1)/2 + a (postcal.cpp:19-59 without U log(1-gamma))."""
    out = []
    for J in range(c + 1):
        for a in range(J + 1):
            v = J * (np.log(g) - np.log1p(-g))
            if p == 1.0:
                v = v if a == J else -np.inf
            elif p != 0.0:
                v += a * np.log(p) + (J - a) * np.log((1 - p) / 2)
            out.append(v)
    return np.array(out)


def ref_totals(tab, U, g, p):
    c = next(k for k in range(9) if ntab(k) == tab.shape[1])
    with np.errstate(invalid="ignore"):
        return U * np.log1p(-g) + logsumexp(log_pi(c, g, p)[None, :] + tab, axis=1)


def ref_joint(tab, U, g, p):
    return float(ref_totals(tab, U, g, p).sum())


def fit(tab, U, how, gamma=0.01, p=0.75):
    import pipsort_b200 as P
    return P.fit_prior(tab, U, fit=how, gamma=gamma, p=p)


def logit(x):
    return np.log(x) - np.log1p(-x)


def expit(u):
    return 1.0 / (1.0 + np.exp(-u))


def ref_fit_p(tab, U, g):
    """The best p in (0, 1) for fixed gamma: a dense grid in log-odds, then bounded Brent around its best point."""
    us = np.linspace(-20, 20, 4001)
    f = [ref_joint(tab, U, g, expit(u)) for u in us]
    k = int(np.argmax(f))
    r = minimize_scalar(lambda u: -ref_joint(tab, U, g, expit(u)), bounds=(us[max(k - 1, 0)], us[min(k + 1, len(us) - 1)]),
                        method="bounded", options=dict(xatol=1e-11))
    return expit(r.x), -r.fun


def ref_fit_gamma_p(tab, U):
    ug, up = np.linspace(-12, 4, 161), np.linspace(-12, 12, 241)
    F = np.array([[ref_joint(tab, U, expit(a), expit(b)) for b in up] for a in ug])
    i, j = np.unravel_index(int(np.argmax(F)), F.shape)
    a, b, best = ug[i], up[j], F[i, j]
    for _ in range(200):
        ra = minimize_scalar(lambda t: -ref_joint(tab, U, expit(t), expit(b)), bounds=(a - 0.2, a + 0.2), method="bounded",
                             options=dict(xatol=1e-11))
        a = ra.x
        rb = minimize_scalar(lambda t: -ref_joint(tab, U, expit(a), expit(t)), bounds=(b - 0.2, b + 0.2), method="bounded",
                             options=dict(xatol=1e-11))
        b = rb.x
        if -rb.fun - best < 1e-13:
            best = max(best, -rb.fun)
            break
        best = -rb.fun
    return expit(a), expit(b), best


def model_tables(n, c, seed):
    """Class tables with the shape of real ones: T[0][0] = 1 (the empty configuration), J >= 1 classes a sum over subsets
    with signals that are shared (favour a = J) or ancestry-specific (favour a = 0) in a locus-dependent mix."""
    rng = np.random.default_rng(seed)
    tab = np.empty((n, ntab(c)))
    for i in range(n):
        s_shared, s_own = rng.uniform(0, 14), rng.uniform(0, 14)
        k = 0
        for J in range(c + 1):
            for a in range(J + 1):
                tab[i, k] = a * s_shared / max(J, 1) * J ** 0.5 + (J - a) * s_own / max(J, 1) * J ** 0.5 + rng.normal(0, 0.3) * (J > 0)
                k += 1
        tab[i] -= rng.uniform(0, 3)            # -K/2
    return tab, rng.integers(2, 30, size=n).astype(np.int32)


# ---- 1. evaluation --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [0, 1, 3, 5, 8])
def test_evaluate_equals_logsumexp(c):
    rng = np.random.default_rng(c)
    tab = rng.uniform(-30, 30, size=(9, ntab(c)))
    tab[rng.random(tab.shape) < 0.2] = -np.inf             # empty classes
    tab[:, 0] = rng.uniform(-5, 0, size=9)                  # the empty configuration is always there
    U = rng.integers(1, 3000, size=9).astype(np.int32)
    for g in (1e-8, 1e-3, 0.01, 0.2, 0.9):
        for p in (0.0, 1e-300, 1e-9, 0.25, 0.75, 0.999999, 1.0):
            g2, p2, joint, per = fit(tab, U, 0, gamma=g, p=p)
            assert (g2, p2) == (g, p)
            want = ref_totals(tab, U, g, p)
            np.testing.assert_allclose(per, want, rtol=1e-13, atol=1e-12, err_msg=f"gamma={g} p={p}")
            assert joint == pytest.approx(per.sum(), rel=1e-15)


def test_p0_is_not_the_limit():
    """p == 0 is the reference's separate prior (no sharing term): not what p -> 0 gives."""
    tab, U = model_tables(5, 3, 1)
    at0 = fit(tab, U, 0, p=0.0)[2]
    near0 = fit(tab, U, 0, p=1e-15)[2]
    assert at0 == pytest.approx(ref_joint(tab, U, 0.01, 0.0), rel=1e-13)
    assert abs(at0 - near0) > 1.0


# ---- 2. fits against scipy ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [3, 11])
def test_fit_p_matches_scipy(seed):
    tab, U = model_tables(30, 3, seed)
    g, p, joint, per = fit(tab, U, "p", gamma=0.01)
    assert g == 0.01
    wp, wf = ref_fit_p(tab, U, 0.01)
    assert 1e-3 < wp < 1 - 1e-3, "the optimum is interior (the test would be weak otherwise)"
    assert abs(p - wp) < 1e-6
    assert joint >= wf - 1e-9
    np.testing.assert_allclose(per, ref_totals(tab, U, g, p), rtol=1e-13)


@pytest.mark.parametrize("seed", [5])
def test_fit_gamma_and_p_matches_scipy(seed):
    tab, U = model_tables(30, 3, seed)
    g, p, joint, _ = fit(tab, U, "gamma,p")
    wg, wp, wf = ref_fit_gamma_p(tab, U)
    assert 1e-3 < wp < 1 - 1e-3 and 1e-6 < wg < 0.5
    assert abs(p - wp) < 1e-6
    assert abs(logit(g) - logit(wg)) < 1e-6
    assert joint >= wf - 1e-9


def test_fit_gamma_only():
    tab, U = model_tables(20, 2, 8)
    g, p, joint, _ = fit(tab, U, "gamma", p=0.4)
    assert p == 0.4
    r = minimize_scalar(lambda u: -ref_joint(tab, U, expit(u), 0.4), bounds=(-18, 18), method="bounded", options=dict(xatol=1e-11))
    assert abs(logit(g) - r.x) < 1e-6
    assert joint >= -r.fun - 1e-9


# ---- 3. documented answers ------------------------------------------------------------------------------------------------
def test_p0_outweighs_every_p_and_is_not_searched():
    """The skip rule weighs every class at least as much as any p in (0, 1] (its three sharing states weigh 1 each): its
    evidence is never smaller, on any locus, so a fit of p leaves it out; gamma is fitted under it when p = 0 is given."""
    tab, U = model_tables(20, 3, 17)
    at0 = fit(tab, U, 0, p=0.0)[3]
    for p in (1e-12, 1e-3, 0.3, 0.75, 0.999, 1.0):
        assert (at0 > fit(tab, U, 0, p=p)[3]).all()
    g, p, _, _ = fit(tab, U, "p")
    assert 0.0 < p <= 1.0
    g, p, _, _ = fit(tab, U, "gamma,p")
    assert 0.0 < p <= 1.0
    g, p, joint, _ = fit(tab, U, "gamma", p=0.0)
    assert p == 0.0
    r = minimize_scalar(lambda u: -ref_joint(tab, U, expit(u), 0.0), bounds=(-18, 18), method="bounded", options=dict(xatol=1e-11))
    assert abs(logit(g) - r.x) < 1e-6
    assert joint >= -r.fun - 1e-9


def test_p1_optimum():
    """Only classes with every SNP shared (a = J) hold anything: the evidence grows with p up to p = 1 itself."""
    tab = np.full((3, ntab(3)), -np.inf)
    for J in range(4):
        tab[:, J * (J + 1) // 2 + J] = 9.0 * J - 1.0
    tab[0, 1] = -1.5                                       # one small ancestry-specific class
    U = np.full(3, 4, dtype=np.int32)
    for how in ("p", "gamma,p"):
        g, p, joint, _ = fit(tab, U, how)
        assert p == 1.0
        assert joint > ref_joint(tab, U, g, 1 - 1e-9)


def bimodal_tables():
    """A locus whose three strong SNPs are either all shared (T[3][3]) or all ancestry-specific (T[3][0]): its evidence
    ~ max(p^3 e^40, ((1-p)/2)^3 e^43) has a maximum at each end; two loci with one shared SNP (~ log p) and one with an
    ancestry-specific SNP (~ log(1-p)) pull both maxima inside: two interior maxima, the higher one (p ~ 0.82) in the
    narrower basin (the trough is at p ~ 0.56)."""
    rows = []
    for cls, v in [((6, 9), (43.0, 40.0)), ((2,), (20.0,)), ((2,), (20.0,)), ((1,), (20.0,))]:
        t = np.full(ntab(3), -np.inf)
        t[0] = 0.0
        t[list(cls)] = v
        rows.append(t)
    return np.array(rows), np.full(len(rows), 30, dtype=np.int32)


def test_bimodal_global_maximum_in_the_narrower_basin():
    tab, U = bimodal_tables()
    us = np.linspace(-25, 25, 20001)
    f = np.array([ref_joint(tab, U, 0.01, expit(u)) for u in us])
    peaks = [k for k in range(1, len(f) - 1) if f[k] > f[k - 1] and f[k] >= f[k + 1]]
    assert len(peaks) == 2, "the objective has two interior maxima"
    trough = peaks[0] + int(np.argmin(f[peaks[0]:peaks[1]]))
    ps = expit(us)
    width = [ps[trough] - 0.0, 1.0 - ps[trough]]          # the basins in p: (0, trough) and (trough, 1)
    k = int(np.argmax(f))
    glob = 0 if k < trough else 1
    assert width[glob] < width[1 - glob], "the global maximum lies in the narrower basin"
    g, p, joint, _ = fit(tab, U, "p")
    r = minimize_scalar(lambda u: -ref_joint(tab, U, 0.01, expit(u)), bounds=(us[k - 1], us[k + 1]), method="bounded",
                        options=dict(xatol=1e-11))
    assert abs(p - expit(r.x)) < 1e-6
    assert joint >= -r.fun - 1e-9


def test_empty_classes():
    """-inf classes (a locus of 2 union SNPs read at c = 3 has no J = 3 class; p = 1 silences a < J) are fitted as any
    other; a locus with no class of non-zero weight at any candidate is refused and named."""
    tab, U = model_tables(12, 3, 21)
    tab[::3, 6:] = -np.inf                                   # J = 3 empty
    tab[1, 1] = tab[1, 3] = tab[1, 4] = -np.inf
    g, p, joint, per = fit(tab, U, "p")
    wp, wf = ref_fit_p(tab, U, 0.01)
    assert abs(p - wp) < 1e-6 and np.isfinite(per).all()
    bad = tab.copy()
    bad[4] = -np.inf
    with pytest.raises(Exception) as ei:
        fit(bad, U, "p")
    assert ei.value.code == PIPSORT_E_ARG and "locus 4" in str(ei.value)
    only_split = np.full((2, ntab(2)), -np.inf)
    only_split[:, 1] = 3.0                                   # J = 1, a = 0 only: zero weight at p = 1
    only_split[0, 0] = 0.0
    U2 = np.array([10, 10], dtype=np.int32)
    with pytest.raises(Exception) as ei:
        fit(only_split, U2, 0, p=1.0)
    assert ei.value.code == PIPSORT_E_ARG and "locus 1" in str(ei.value)
    assert fit(only_split, U2, "p")[1] < 1.0


# ---- 4. refusals ----------------------------------------------------------------------------------------------------------
def call(n_loci=2, c=1, tab=None, U=(5, 5), fitbits=2, gamma=0.01, p=0.5):
    import pipsort_b200 as P
    from pipsort_b200.engine import _dp
    tab = np.zeros((2, ntab(max(c, 0)))) if tab is None else tab
    Ua = np.ascontiguousarray(U, dtype=np.int32)
    g, q, j = C.c_double(gamma), C.c_double(p), C.c_double()
    rc = P.lib().pipsort_fit_prior(n_loci, c, _dp(np.ascontiguousarray(tab, dtype=np.float64)), Ua.ctypes.data_as(C.POINTER(C.c_int32)),
                                   fitbits, C.byref(g), C.byref(q), C.byref(j), None)
    return rc, P.lib().pipsort_last_error().decode()


def nan_table():
    t = np.zeros((2, 3))
    t[1, 2] = np.nan
    return t


def inf_table():
    t = np.zeros((2, 3))
    t[0, 1] = np.inf
    return t


@pytest.mark.parametrize("kw,text", [(dict(n_loci=0), "n_loci=0"), (dict(n_loci=-2), "n_loci=-2"), (dict(c=9), "c=9"),
                                     (dict(c=-1), "c=-1"), (dict(fitbits=4), "fit=4"), (dict(gamma=0.0), "gamma=0"),
                                     (dict(gamma=1.0), "gamma=1"), (dict(gamma=float("nan")), "gamma=nan"),
                                     (dict(p=-0.1), "sharing_param=-0.1"), (dict(p=1.5), "sharing_param=1.5"),
                                     (dict(U=(5, 0)), "union_count[1]=0"), (dict(U=(-3, 5)), "union_count[0]=-3"),
                                     (dict(tab=nan_table()), "tables[1][2]=nan"), (dict(tab=inf_table()), "tables[0][1]=inf")])
def test_refusals_name_the_value(kw, text):
    rc, msg = call(**kw)
    assert rc == PIPSORT_E_ARG
    assert text in msg, msg


def test_python_refusals():
    import pipsort_b200 as P
    with pytest.raises(ValueError):
        P.fit_prior(np.zeros((2, 4)), [1, 1])             # 4 is no (c+1)(c+2)/2
    with pytest.raises(ValueError):
        P.fit_prior(np.zeros((2, 3)), [1])
    with pytest.raises(ValueError):
        P.fit_prior(np.zeros((2, 3)), [1, 1], fit="q")
    with pytest.raises(ValueError):
        P.LocusBatch([], 3, priors=[(0.01, 0.5)], class_evidence=True)
    assert P.class_evidence_batch([], 3).shape == (0, 10)
    with pytest.raises(P.PipsortError) as ei:
        P.class_evidence_batch([], 9)
    assert ei.value.code == PIPSORT_E_ARG and "c=9" in str(ei.value)
