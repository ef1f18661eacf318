"""Host-side phases of pipsort_create inside the one-locus call (PIPSORT_TRACE_CREATE=1): python scripts/one_call_trace.py.
The create / run / read / destroy phases of a locus are timed through the engine API by scripts/e2e_breakdown.py."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import pipsort_b200 as P
from pipsort_b200 import synth
L = synth.make_locus(150)
sig = np.concatenate([s.ravel() for s in L.sigma]); z = np.concatenate(L.z)
for _ in range(6):
    P.posterior_exhaustive(L.num_snps, sig, z, L.d, L.K, L.snp_map, 3, gamma=L.gamma, sharing_param=L.sharing_param)
