"""pipsort_posterior_exhaustive_grid_batch refuses bad arguments and bad priors before it touches CUDA (no device needed)."""
import ctypes as C

import numpy as np
import pytest

PIPSORT_E_ARG = 1


def call(n_loci=1, loci=True, outs=True, priors=((0.01, 0.75),), gamma=True, sharing=True, n_priors=None):
    import pipsort_b200 as P
    from pipsort_b200.engine import _LocusV, _OutputsV, _dp
    lib = P.lib()
    pr = np.asarray(priors, dtype=np.float64).reshape(-1, 2)
    gam, p = np.ascontiguousarray(pr[:, 0]), np.ascontiguousarray(pr[:, 1])
    la = (_LocusV * max(n_loci, 1))()          # never read: every call below fails or returns before the loci are used
    oa = (_OutputsV * max(n_loci * len(pr), 1))()
    cnt = (C.c_uint64 * max(n_loci, 1))()
    rc = lib.pipsort_posterior_exhaustive_grid_batch(la if loci else None, n_loci, 0, 0, 3,
                                                     len(pr) if n_priors is None else n_priors,
                                                     _dp(gam) if gamma else None, _dp(p) if sharing else None,
                                                     oa if outs else None, cnt)
    return rc, lib.pipsort_last_error().decode()


@pytest.mark.parametrize("kw", [dict(n_loci=-1), dict(loci=False), dict(outs=False), dict(gamma=False), dict(sharing=False),
                                dict(n_priors=0), dict(n_priors=-3), dict(priors=())])
def test_bad_arguments(kw):
    rc, _ = call(**kw)
    assert rc == PIPSORT_E_ARG


@pytest.mark.parametrize("bad,what", [((1.0, 0.5), "gamma"), ((0.0, 0.5), "gamma"), ((0.01, 1.5), "sharing_param"),
                                      ((0.01, -0.1), "sharing_param"), ((float("nan"), 0.5), "gamma"),
                                      ((0.01, float("nan")), "sharing_param")])
def test_bad_prior_is_named(bad, what):
    """The bad prior is found before any engine exists, whatever the loci (here: never read), and its index is named."""
    for n_loci in (0, 40):
        rc, msg = call(n_loci=n_loci, priors=[(0.01, 0.75), (0.2, 0.25), bad])
        assert rc == PIPSORT_E_ARG
        assert "prior 2" in msg and what in msg


def test_no_loci_returns_zero():
    assert call(n_loci=0)[0] == 0
    assert call(n_loci=0, loci=False, outs=False)[0] == 0


def test_python_refusals():
    import pipsort_b200 as P
    with pytest.raises(ValueError):
        P.LocusBatch([], 3, evidence_only=True)
    B = P.LocusBatch([], 3, priors=[(0.01, 0.75)], evidence_only=True).run()
    assert B.evidence().shape == (0, 1, 3)
    with pytest.raises(P.PipsortError) as ei:
        P.posterior_exhaustive_grid_batch([], 3, [(0.01, 0.75), (1.0, 0.5)])
    assert ei.value.code == PIPSORT_E_ARG and "prior 1" in str(ei.value)
