"""pipsort_sss_batch refuses bad arguments, and loci the search cannot run on, before it touches CUDA (no device needed).
A refusal of one locus names it."""
import ctypes as C

import numpy as np
import pytest

PIPSORT_E_ARG, PIPSORT_E_RANGE = 1, 4
PRIOR_CLASSES, CAUSAL_COUNTS = 8, 16
SSS_MAX_U = (1 << 15) - 2


def call(n_loci=1, loci=True, outs=True, flags=0, c=3, max_iterations=1000, bad=None):
    """The C-ABI call on n_loci locus structs of which only union_count and sharing_param are set (U = 10, p = 0.75): every
    call below is refused or returns before any other field is read.  bad = (i, U, p) sets locus i."""
    import pipsort_b200 as P
    from pipsort_b200.engine import _LocusV, _OutputsV
    lib = P.lib()
    la = (_LocusV * max(n_loci, 1))()
    for i in range(n_loci):
        la[i].union_count, la[i].sharing_param = 10, 0.75
    if bad is not None:
        i, U, p = bad
        la[i].union_count, la[i].sharing_param = U, p
    oa = (_OutputsV * max(n_loci, 1))()
    it = (C.c_int32 * max(n_loci, 1))()
    why = (C.c_int32 * max(n_loci, 1))()
    cnt = (C.c_uint64 * max(n_loci, 1))()
    rc = lib.pipsort_sss_batch(la if loci else None, n_loci, 0, flags, c, max_iterations, oa if outs else None, it, why, cnt)
    return rc, lib.pipsort_last_error().decode()


@pytest.mark.parametrize("kw", [dict(n_loci=-1), dict(loci=False), dict(outs=False),
                                dict(n_loci=0, c=-1), dict(n_loci=40, c=-1), dict(n_loci=0, c=9), dict(n_loci=40, c=9),
                                dict(n_loci=0, max_iterations=-1), dict(n_loci=40, max_iterations=-1),
                                dict(flags=PRIOR_CLASSES), dict(flags=CAUSAL_COUNTS), dict(n_loci=0, flags=PRIOR_CLASSES)])
def test_bad_arguments(kw):
    """Refused whether the list is empty or not."""
    rc, _ = call(**kw)
    assert rc == PIPSORT_E_ARG


def test_classes_refusal_says_why():
    rc, msg = call(flags=PRIOR_CLASSES)
    assert rc == PIPSORT_E_ARG and "PIPSORT_PRIOR_CLASSES" in msg


@pytest.mark.parametrize("U,p,c,code,text", [(10, 1.0, 3, PIPSORT_E_ARG, "sharing_param = 1"),
                                             (10, 1.0, 1, PIPSORT_E_ARG, "sharing_param = 1"),
                                             (SSS_MAX_U + 1, 0.75, 3, PIPSORT_E_RANGE, "15 bits"),
                                             (SSS_MAX_U + 1, 0.75, 0, PIPSORT_E_RANGE, "15 bits")])
def test_bad_locus_is_named(U, p, c, code, text):
    """Locus 17 of 40 is refused with the code pipsort_sss returns for it, before any engine exists, and the message names
    it; so is locus 0 of 1."""
    for n_loci, i in ((40, 17), (1, 0)):
        rc, msg = call(n_loci=n_loci, c=c, bad=(i, U, p))
        assert rc == code, msg
        assert msg.startswith(f"locus {i}: ") and text in msg


def test_no_loci_returns_zero():
    assert call(n_loci=0)[0] == 0
    assert call(n_loci=0, loci=False, outs=False)[0] == 0


def test_python_refusals():
    import pipsort_b200 as P
    with pytest.raises(ValueError):
        P.LocusBatch([], 3, search=True, priors=[(0.01, 0.75)])
    with pytest.raises(ValueError):
        P.LocusBatch([], 3, search=True, class_evidence=True)
    res, it, why = P.sss_batch([], 3)
    assert res == [] and it.shape == (0,) and why.shape == (0,)
    for c, mi in ((9, 10), (-1, 10), (3, -1)):
        with pytest.raises(P.PipsortError) as ei:
            P.sss_batch([], c, max_iterations=mi)
        assert ei.value.code == PIPSORT_E_ARG


def test_python_names_the_locus():
    """sss_batch marshals the loci through LocusBatch: the refusal of locus 17 of 40 reaches the caller with its index."""
    import pipsort_b200 as P
    L = dict(num_snps=np.array([2, 2], dtype=np.int32), sigma=np.concatenate([np.eye(2).ravel()] * 2), z=np.zeros(4),
             d=np.array([5.0, 5.0]), K=0.0, snp_map=np.array([[0, 1], [0, 1]], dtype=np.int32), gamma=0.01, sharing_param=0.75)
    loci = [dict(L) for _ in range(40)]
    loci[17]["sharing_param"] = 1.0
    with pytest.raises(P.PipsortError) as ei:
        P.sss_batch(loci, 2)
    assert ei.value.code == PIPSORT_E_ARG and "locus 17: " in str(ei.value)
