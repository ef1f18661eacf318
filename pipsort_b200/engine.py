"""ctypes binding of the C-ABI in include/pipsort_b200.h (the engine itself is CUDA, csrc/).

`Engine` mirrors the part of the reference's PostCal class that is the hot path (postcal.h:118-195,
postcal.cpp:716-1092, sss_postcal.cpp:447-685): construct it from what the PostCal constructor
receives, call compute_total_likelihood() / score_union_configs(), read the same result arrays.
There is no CPU path: the library must load and a CUDA device must be present.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from . import build as _build

_lib = None

KEEP_ORDER = 1
GENERIC_ONLY = 2
RAW_LD = 4
PRIOR_CLASSES = 8
CAUSAL_COUNTS = 16
IPC_HANDLE_BYTES = 64
KMAX = 8


class PipsortError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"pipsort_b200 error {code}: {msg}")
        self.code = code


class _Locus(C.Structure):
    _fields_ = [("num_studies", C.c_int32), ("num_snps", C.POINTER(C.c_int32)), ("sigma", C.POINTER(C.c_double)),
                ("z", C.POINTER(C.c_double)), ("d", C.POINTER(C.c_double)), ("K", C.c_double),
                ("union_count", C.c_int32), ("snp_map", C.POINTER(C.c_int32)), ("gamma", C.c_double),
                ("sharing_param", C.c_double), ("max_causal", C.c_int32)]


class _LocusV(C.Structure):      # same layout as _Locus with untyped pointers: filled from ndarray.ctypes.data (cheap)
    _fields_ = [("num_studies", C.c_int32), ("num_snps", C.c_void_p), ("sigma", C.c_void_p), ("z", C.c_void_p),
                ("d", C.c_void_p), ("K", C.c_double), ("union_count", C.c_int32), ("snp_map", C.c_void_p),
                ("gamma", C.c_double), ("sharing_param", C.c_double), ("max_causal", C.c_int32)]


class _OutputsV(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("total", "postValues", "noCausal", "sharedPips", "sharedLL", "notSharedLL")]


class _PrepInfo(C.Structure):
    _fields_ = [("add_diag", C.c_double), ("K", C.c_double), ("min_abs_eig", C.c_double), ("n_negative", C.c_int32),
                ("psd_iterations", C.c_int32)]


class _Outputs(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_double)) for n in
                ("total", "postValues", "noCausal", "sharedPips", "sharedLL", "notSharedLL")]


def lib():
    """Loads pipsort_b200/lib/libpipsort_b200.so (builds it first if the sources are newer)."""
    global _lib
    if _lib is None:
        path = _build.build_engine()          # rebuilds only when the library is missing or its sources changed (content hash)
        L = C.CDLL(path)
        vp, u64, i32 = C.c_void_p, C.c_uint64, C.c_int
        L.pipsort_create.argtypes = [C.POINTER(_Locus), i32, C.c_uint32, C.POINTER(vp)]
        L.pipsort_preprocess_study.argtypes = [i32, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                               C.POINTER(C.c_double), C.POINTER(_PrepInfo)]
        L.pipsort_prep_info_get.argtypes = [vp, i32, C.POINTER(_PrepInfo)]
        L.pipsort_posterior_exhaustive.argtypes = [C.POINTER(_LocusV), i32, C.c_uint32, i32, C.POINTER(_OutputsV), C.POINTER(u64)]
        L.pipsort_posterior_exhaustive_batch.argtypes = [C.POINTER(_LocusV), C.c_int32, i32, C.c_uint32, i32,
                                                         C.POINTER(_OutputsV), C.POINTER(u64)]
        L.pipsort_posterior_exhaustive_grid_batch.argtypes = [C.POINTER(_LocusV), C.c_int32, i32, C.c_uint32, i32, i32,
                                                              C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_OutputsV),
                                                              C.POINTER(u64)]
        L.pipsort_read_class_evidence.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(u64)]
        L.pipsort_class_evidence_batch.argtypes = [C.POINTER(_LocusV), C.c_int32, i32, C.c_uint32, i32, C.POINTER(C.c_double),
                                                   C.POINTER(u64)]
        L.pipsort_read_count_table.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(u64)]
        L.pipsort_count_table_batch.argtypes = [C.POINTER(_LocusV), C.c_int32, i32, C.c_uint32, i32, C.POINTER(C.c_double),
                                                C.POINTER(u64)]
        L.pipsort_count_posterior.argtypes = [C.c_int32, i32, C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_double,
                                              C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.pipsort_fit_prior.argtypes = [C.c_int32, i32, C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_uint32,
                                        C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.pipsort_destroy.argtypes = [vp]
        L.pipsort_destroy.restype = None
        L.pipsort_reset.argtypes = [vp]
        L.pipsort_total_ranks.argtypes = [vp, i32, C.POINTER(u64)]
        L.pipsort_run_exhaustive.argtypes = [vp, i32, u64, u64]
        L.pipsort_score_union_configs.argtypes = [vp, C.POINTER(C.c_int32), C.c_int64, i32, C.POINTER(C.c_uint8),
                                                  C.POINTER(C.c_double)]
        L.pipsort_score_union_configs_device.argtypes = [vp, vp, C.c_int64, i32, vp, vp]
        L.pipsort_score_given_configs.argtypes = [vp, C.POINTER(C.c_int16), C.c_int64, i32]
        L.pipsort_score_given_configs_device.argtypes = [vp, vp, C.c_int64, i32]
        L.pipsort_sss.argtypes = [vp, i32, i32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.pipsort_sss_reset.argtypes = [vp]
        L.pipsort_sss_sharded.argtypes = [vp, i32, i32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.pipsort_sss_batch.argtypes = [C.POINTER(_LocusV), C.c_int32, i32, C.c_uint32, i32, i32, C.POINTER(_OutputsV),
                                        C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(u64)]
        L.pipsort_read_accumulators.argtypes = [vp, C.POINTER(_Outputs)]
        L.pipsort_read_prior_grid.argtypes = [vp, i32, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_OutputsV),
                                              C.POINTER(u64)]
        L.pipsort_posterior_exhaustive_grid.argtypes = [C.POINTER(_LocusV), i32, C.c_uint32, i32, i32, C.POINTER(C.c_double),
                                                        C.POINTER(C.c_double), C.POINTER(_OutputsV), C.POINTER(u64)]
        L.pipsort_finalize.argtypes = [vp]
        L.pipsort_finalize_reset.argtypes = [vp]
        L.pipsort_fetch_results.argtypes = [vp, C.POINTER(_Outputs)]
        L.pipsort_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.pipsort_config_count.argtypes = [vp, C.POINTER(u64)]
        L.pipsort_last_read_config_count.argtypes = [vp, C.POINTER(u64)]
        L.pipsort_enumerate.argtypes = [vp, i32, u64, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                        C.POINTER(C.c_uint32)]
        L.pipsort_accumulator_buffer.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
        L.pipsort_merge.argtypes = [vp, vp]
        L.pipsort_shard_ranks.argtypes = [vp, i32, i32, C.POINTER(u64)]
        L.pipsort_graph_begin.argtypes = [vp]
        L.pipsort_graph_end.argtypes = [vp, C.POINTER(C.c_int32)]
        L.pipsort_graph_launch.argtypes = [vp, C.c_int32]
        L.pipsort_p2p_export.argtypes = [vp, i32, C.c_char_p]
        L.pipsort_p2p_connect.argtypes = [vp, C.c_char_p, i32, i32, i32]
        L.pipsort_p2p_reduce_to_root.argtypes = [vp]
        L.pipsort_p2p_reduce_to_root_reset.argtypes = [vp]
        L.pipsort_p2p_combine_finalize.argtypes = [vp]
        L.pipsort_shard_ranks_for_map.argtypes = [C.POINTER(C.c_int32), C.c_int32, i32, i32, C.c_uint32, C.POINTER(u64)]
        L.pipsort_stream.argtypes = [vp]
        L.pipsort_stream.restype = vp
        L.pipsort_sync.argtypes = [vp]
        L.pipsort_set_stream.argtypes = [vp, vp]
        L.pipsort_flush_l2.argtypes = [vp]
        L.pipsort_timer_begin.argtypes = [vp]
        L.pipsort_timer_end.argtypes = [vp, C.POINTER(C.c_float)]
        L.pipsort_launch_count.argtypes = [vp]
        L.pipsort_launch_count.restype = u64
        L.pipsort_measure_fp64_peak.argtypes = [i32, C.POINTER(C.c_double)]
        L.pipsort_last_error.restype = C.c_char_p
        L.pipsort_version.restype = C.c_char_p
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise PipsortError(rc, lib().pipsort_last_error().decode())


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


@dataclass
class Results:
    """PostCal's result members (postcal.h:62-99): log space, 0.0 = nothing accumulated."""
    total: float
    postValues: np.ndarray
    noCausal: np.ndarray
    sharedPips: np.ndarray
    sharedLL: np.ndarray
    notSharedLL: np.ndarray
    n_configs: int = 0

    @staticmethod
    def _special_exp(x, total):           # postcal.h:277-283
        with np.errstate(over="ignore"):
            return np.where(x == 0, 0.0, np.exp(x - total))

    def pips(self):
        return self._special_exp(self.postValues, self.total)

    def shared_pips(self):
        return self._special_exp(self.sharedPips, self.total)

    def no_causal(self):
        return self._special_exp(self.noCausal, self.total)


class Engine:
    """Device-resident locus + accumulators (the hot-path half of the reference's PostCal)."""

    def __init__(self, num_snps, sigma, z, d, K, snp_map, gamma=0.01, sharing_param=0.75, max_causal=3, device=0,
                 keep_order=False, generic_only=False, raw_ld=False, prior_classes=False, causal_counts=False):
        self.num_snps = np.ascontiguousarray(num_snps, dtype=np.int32)
        if isinstance(sigma, (list, tuple)):
            sigma = np.concatenate([np.asarray(s, dtype=np.float64).ravel() for s in sigma])
        if isinstance(z, (list, tuple)):
            z = np.concatenate([np.asarray(v, dtype=np.float64).ravel() for v in z])
        sigma = np.ascontiguousarray(sigma, dtype=np.float64).ravel()
        z = np.ascontiguousarray(z, dtype=np.float64).ravel()
        d = np.ascontiguousarray(d, dtype=np.float64)
        smap = np.ascontiguousarray(snp_map, dtype=np.int32)
        self.S = len(self.num_snps)
        self.U = int(smap.shape[1]) if smap.ndim == 2 else 0
        self.N = int(self.num_snps.sum())
        assert sigma.size == int((self.num_snps.astype(np.int64) ** 2).sum()), "sigma size"
        assert z.size == self.N, "z size"
        loc = _Locus(self.S, self.num_snps.ctypes.data_as(C.POINTER(C.c_int32)), _dp(sigma), _dp(z), _dp(d), float(K),
                     self.U, smap.ctypes.data_as(C.POINTER(C.c_int32)), float(gamma), float(sharing_param),
                     int(max_causal))
        self._h = C.c_void_p()
        _check(lib().pipsort_create(C.byref(loc), int(device), (KEEP_ORDER if keep_order else 0) | (GENERIC_ONLY if generic_only else 0) |
                                    (RAW_LD if raw_ld else 0) | (PRIOR_CLASSES if prior_classes else 0) |
                                    (CAUSAL_COUNTS if causal_counts else 0), C.byref(self._h)))
        self.max_causal = int(max_causal)
        self.device = int(device)

    def prep_info(self, study):
        """What the on-device pre-processing found (engines created with raw_ld=True): dict of pipsort_prep_info."""
        info = _PrepInfo()
        _check(lib().pipsort_prep_info_get(self._h, int(study), C.byref(info)))
        return {k: getattr(info, k) for k, _ in _PrepInfo._fields_}

    # -- lifetime ------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().pipsort_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- the hot path ----------------------------------------------------------------------------------
    def reset(self):
        _check(lib().pipsort_reset(self._h))

    def total_ranks(self, c):
        out = C.c_uint64()
        _check(lib().pipsort_total_ranks(self._h, int(c), C.byref(out)))
        return int(out.value)

    def run_exhaustive(self, c, rank_begin=0, rank_end=None):
        """computeTotalLikelihood (postcal.cpp:716) over union-subset ranks [rank_begin, rank_end); asynchronous."""
        if rank_end is None:
            rank_end = self.total_ranks(c)
        _check(lib().pipsort_run_exhaustive(self._h, int(c), int(rank_begin), int(rank_end)))

    def compute_total_likelihood(self, c=None):
        """The reference's PostCal::computeTotalLikelihood: whole rank space, returns the results."""
        c = self.max_causal if c is None else c
        self.reset()
        self.run_exhaustive(c)
        return self.read()

    def score_union_configs(self, idx, make_updates=None):
        """expand_and_compute_lkl (sss_postcal.cpp:447) for a batch; returns max-|l| expansion per configuration."""
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        if idx.ndim == 1:
            idx = idx.reshape(-1, 1)
        n, kmax = idx.shape
        out = np.zeros(n, dtype=np.float64)
        mu = None
        if make_updates is not None:
            mu = np.ascontiguousarray(make_updates, dtype=np.uint8)
            assert mu.size == n
        _check(lib().pipsort_score_union_configs(
            self._h, idx.ctypes.data_as(C.POINTER(C.c_int32)), n, kmax,
            mu.ctypes.data_as(C.POINTER(C.c_uint8)) if mu is not None else None, _dp(out)))
        return out

    def score_union_configs_device(self, d_idx_ptr, n, kmax, d_upd_ptr, d_out_ptr):
        _check(lib().pipsort_score_union_configs_device(self._h, C.c_void_p(d_idx_ptr), int(n), int(kmax),
                                                        C.c_void_p(d_upd_ptr), C.c_void_p(d_out_ptr)))

    def score_given_configs(self, configs):
        """computeTotalLikelihoodGivenConfigs (postcal.cpp:400-714, -b/-d/-e): int16[num_configs][num_groups] of global
        SNP indices, negative = unused group; accumulates (call reset() first for a fresh PostCal)."""
        cfg = np.ascontiguousarray(configs, dtype=np.int16)
        if cfg.ndim != 2:
            raise ValueError("configs must be a num_configs x num_groups matrix")
        _check(lib().pipsort_score_given_configs(self._h, cfg.ctypes.data_as(C.POINTER(C.c_int16)), cfg.shape[0],
                                                 cfg.shape[1]))

    def compute_total_likelihood_given_configs(self, configs):
        self.reset()
        self.score_given_configs(configs)
        return self.read()

    def sss(self, c=None, max_iterations=1000):
        """sss_computeTotalLikelihood (sss_postcal.cpp:102-380): the whole stochastic shotgun search on a fresh set of
        accumulators.  Returns (Results, iterations, stop_reason) with stop_reason 0 = iteration cap, 1 = no new
        configuration ("hit break condition"), 2 = convergence."""
        c = self.max_causal if c is None else c
        it, why = C.c_int32(), C.c_int32()
        self.reset()
        _check(lib().pipsort_sss(self._h, int(c), int(max_iterations), C.byref(it), C.byref(why)))
        return self.read(), int(it.value), int(why.value)

    def sss_sharded(self, c=None, max_iterations=1000):
        """pipsort_sss_sharded: the search with every neighbourhood split over the ranks of the p2p group (call on every
        rank after p2p_connect, on fresh accumulators).  The accumulators stay rank-partial: follow with
        p2p_reduce_to_root() and read() on the root.  Returns (iterations, stop_reason)."""
        c = self.max_causal if c is None else c
        it, why = C.c_int32(), C.c_int32()
        _check(lib().pipsort_sss_sharded(self._h, int(c), int(max_iterations), C.byref(it), C.byref(why)))
        return int(it.value), int(why.value)

    def read(self) -> Results:
        return self._read(lib().pipsort_read_accumulators)

    def _read(self, fn) -> Results:
        total = np.zeros(1)
        post = np.zeros(self.N)
        nc = np.zeros(self.S)
        sp = np.zeros(self.U)
        sl = np.zeros(self.U)
        nl = np.zeros(self.U)
        o = _Outputs(_dp(total), _dp(post), _dp(nc), _dp(sp), _dp(sl), _dp(nl))
        _check(fn(self._h, C.byref(o)))
        cnt = C.c_uint64()
        _check(lib().pipsort_last_read_config_count(self._h, C.byref(cnt)))
        return Results(float(total[0]), post, nc, sp, sl, nl, int(cnt.value))

    def read_prior_grid(self, priors, evidence_only=False):
        """Results for every prior (gamma, p) of `priors` from the accumulators of ONE pass (an engine created with
        prior_classes=True): each equals what an engine created with that prior reports (pipsort_read_prior_grid).
        evidence_only=True: the evidence read, an ndarray [n_priors, 3] of (total, noCausal[0], noCausal[1])."""
        gam, p = _prior_arrays(priors)
        cnt = C.c_uint64()
        if evidence_only:
            ev = np.zeros((len(gam), 3))
            outs = _evidence_outputs(ev)
            _check(lib().pipsort_read_prior_grid(self._h, len(gam), _dp(gam), _dp(p), outs, C.byref(cnt)))
            return ev
        outs, res = _grid_outputs(len(gam), self.N, self.S, self.U)
        _check(lib().pipsort_read_prior_grid(self._h, len(gam), _dp(gam), _dp(p), outs, C.byref(cnt)))
        return res(int(cnt.value))

    def read_class_evidence(self, c):
        """The class table of the store (an engine created with prior_classes=True; pipsort_read_class_evidence): ndarray
        [(c+1)(c+2)/2], entry J(J+1)/2 + a = -K/2 + log T[J][a], -inf for an empty class.  fit_prior takes it."""
        tab = np.empty(_ntab(c))
        _check(lib().pipsort_read_class_evidence(self._h, int(c), _dp(tab), None))
        return tab

    def read_count_table(self, c):
        """The count table of the store (an engine created with causal_counts=True; pipsort_read_count_table): ndarray
        [C(c+3, 3)], entry cnt_idx(J, a, b0) = J(J+1)(J+2)/6 + a(2J+3-a)/2 + b0 = -K/2 + log R[a][b0][b1] (a SNPs causal in
        both studies, b0 in study 0 only, b1 = J - a - b0 in study 1 only), -inf for an empty class.  count_posterior takes
        it; class_tables_from_counts turns it into read_class_evidence's table."""
        tab = np.empty(_ncnt(c))
        _check(lib().pipsort_read_count_table(self._h, int(c), _dp(tab), None))
        return tab

    def finalize(self, reset=False):
        """Bins -> log-space results on the device; reset=True also leaves the accumulators empty (no reset() needed before
        the next pass; fetch() then returns the results)."""
        _check(lib().pipsort_finalize_reset(self._h) if reset else lib().pipsort_finalize(self._h))

    def fetch(self) -> Results:
        """The results of the last finalize (device -> host), without touching the accumulators."""
        return self._read(lib().pipsort_fetch_results)

    def last_kernel_ms(self):
        ms = C.c_float()
        _check(lib().pipsort_last_kernel_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def config_count(self):
        out = C.c_uint64()
        _check(lib().pipsort_config_count(self._h, C.byref(out)))
        return int(out.value)

    def enumerate(self, c, rank, expansion=0):
        idx = np.full(max(c, 1), -1, dtype=np.int32)
        st = np.zeros(max(c, 1), dtype=np.int32)
        ne = C.c_uint32()
        _check(lib().pipsort_enumerate(self._h, int(c), int(rank), int(expansion),
                                       idx.ctypes.data_as(C.POINTER(C.c_int32)),
                                       st.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(ne)))
        k = int((idx[:c] >= 0).sum())
        return idx[:k].tolist(), st[:k].tolist(), int(ne.value)

    # -- multi-GPU plumbing ------------------------------------------------------------------------------
    def accumulator_buffer(self):
        p = C.c_void_p()
        n = C.c_uint64()
        _check(lib().pipsort_accumulator_buffer(self._h, C.byref(p), C.byref(n)))
        return int(p.value), int(n.value)

    def merge_from(self, other: "Engine"):
        _check(lib().pipsort_merge(self._h, other._h))

    def graph_begin(self):
        _check(lib().pipsort_graph_begin(self._h))

    def graph_end(self) -> int:
        gid = C.c_int32()
        _check(lib().pipsort_graph_end(self._h, C.byref(gid)))
        return int(gid.value)

    def graph_launch(self, graph_id):
        _check(lib().pipsort_graph_launch(self._h, int(graph_id)))

    def p2p_export(self, world) -> bytes:
        """CUDA IPC handle of this engine's mailbox (64 bytes; one inbox slot per rank of a group of `world`)."""
        buf = C.create_string_buffer(IPC_HANDLE_BYTES)
        _check(lib().pipsort_p2p_export(self._h, int(world), buf))
        return buf.raw

    def p2p_connect(self, handles, rank, root=0):
        """handles: list of every rank's p2p_export() bytes, in rank order."""
        blob = b"".join(handles)
        assert len(blob) == IPC_HANDLE_BYTES * len(handles)
        _check(lib().pipsort_p2p_connect(self._h, blob, len(handles), int(rank), int(root)))

    def p2p_reduce_to_root(self, reset_sender=False):
        _check(lib().pipsort_p2p_reduce_to_root_reset(self._h) if reset_sender else lib().pipsort_p2p_reduce_to_root(self._h))

    def p2p_combine_finalize(self):
        """Tail of a repeatable multi-GPU pass, one launch per rank (pipsort_p2p_combine_finalize); fetch() on the root."""
        _check(lib().pipsort_p2p_combine_finalize(self._h))

    def shard_ranks(self, c, parts):
        b = (C.c_uint64 * (parts + 1))()
        _check(lib().pipsort_shard_ranks(self._h, int(c), int(parts), b))
        return [int(x) for x in b]

    def stream(self):
        return int(lib().pipsort_stream(self._h) or 0)

    def sync(self):
        _check(lib().pipsort_sync(self._h))

    def set_stream(self, cuda_stream):
        _check(lib().pipsort_set_stream(self._h, C.c_void_p(cuda_stream or None)))

    def flush_l2(self):
        _check(lib().pipsort_flush_l2(self._h))

    def accumulator_tensor(self):
        """Zero-copy torch view of the accumulator store (for torch.distributed all_reduce)."""
        import torch
        ptr, n = self.accumulator_buffer()

        class _View:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}

        return torch.as_tensor(_View(), device=f"cuda:{self.device}")

    def timer_begin(self):
        _check(lib().pipsort_timer_begin(self._h))

    def timer_end(self):
        ms = C.c_float()
        _check(lib().pipsort_timer_end(self._h, C.byref(ms)))
        return float(ms.value)

    def launch_count(self):
        return int(lib().pipsort_launch_count(self._h))


def posterior_exhaustive(num_snps, sigma, z, d, K, snp_map, c, gamma=0.01, sharing_param=0.75, device=0, raw_ld=False):
    """One locus, one call (pipsort_posterior_exhaustive): host arrays in, Results out -- what Model::run does with a fresh
    PostCal.  sigma / z: flat float64 arrays, studies concatenated (or lists of per-study arrays)."""
    num_snps = np.ascontiguousarray(num_snps, dtype=np.int32)
    if isinstance(sigma, (list, tuple)):
        sigma = np.concatenate([np.asarray(s, dtype=np.float64).ravel() for s in sigma])
    if isinstance(z, (list, tuple)):
        z = np.concatenate([np.asarray(v, dtype=np.float64).ravel() for v in z])
    sigma = np.ascontiguousarray(sigma, dtype=np.float64).ravel()
    z = np.ascontiguousarray(z, dtype=np.float64).ravel()
    d = np.ascontiguousarray(d, dtype=np.float64)
    smap = np.ascontiguousarray(snp_map, dtype=np.int32)
    S, U, N = len(num_snps), int(smap.shape[1]), int(num_snps.sum())
    loc = _LocusV(S, num_snps.ctypes.data, sigma.ctypes.data, z.ctypes.data, d.ctypes.data, float(K), U, smap.ctypes.data,
                  float(gamma), float(sharing_param), int(c))
    buf = np.zeros(1 + N + S + 3 * U)
    total, post, nc = buf[0:1], buf[1:1 + N], buf[1 + N:1 + N + S]
    sp, sl, nl = buf[1 + N + S:1 + N + S + U], buf[1 + N + S + U:1 + N + S + 2 * U], buf[1 + N + S + 2 * U:]
    b0 = buf.ctypes.data
    o = _OutputsV(b0, b0 + 8, b0 + 8 * (1 + N), b0 + 8 * (1 + N + S), b0 + 8 * (1 + N + S + U), b0 + 8 * (1 + N + S + 2 * U))
    cnt = C.c_uint64()
    _check(lib().pipsort_posterior_exhaustive(C.byref(loc), int(device), RAW_LD if raw_ld else 0, int(c), C.byref(o), C.byref(cnt)))
    return Results(float(total[0]), post, nc, sp, sl, nl, int(cnt.value))


def _ntab(c):
    """Entries of a class table up to class limit c (0 for a c the engine refuses)."""
    return max(0, (int(c) + 1) * (int(c) + 2) // 2)


def _ncnt(c):
    """Entries of a count table up to class limit c: C(c+3, 3) (0 for a c the engine refuses)."""
    return max(0, (int(c) + 1) * (int(c) + 2) * (int(c) + 3) // 6)


def _cnt_classes(c):
    """(J, a, b0, b1) of every entry of a count table up to c, in table order."""
    return [(J, a, b0, J - a - b0) for J in range(c + 1) for a in range(J + 1) for b0 in range(J - a + 1)]


def _prior_arrays(priors):
    pr = np.asarray(priors, dtype=np.float64).reshape(-1, 2) if len(priors) else np.zeros((0, 2))
    return np.ascontiguousarray(pr[:, 0]), np.ascontiguousarray(pr[:, 1])


def _grid_outputs(n, N, S, U):
    """pipsort_outputs[n] over one buffer, and a function that slices the buffer into Results once it is filled."""
    w = 1 + N + S + 3 * U
    buf = np.zeros((max(n, 1), w))
    outs = (_OutputsV * max(n, 1))()
    for i in range(n):
        b0 = buf[i].ctypes.data
        outs[i] = _OutputsV(b0, b0 + 8, b0 + 8 * (1 + N), b0 + 8 * (1 + N + S), b0 + 8 * (1 + N + S + U), b0 + 8 * (1 + N + S + 2 * U))

    def results(cnt):
        out = []
        for i in range(n):
            r = buf[i]
            p2 = 1 + N + S
            out.append(Results(float(r[0]), r[1:1 + N], r[1 + N:p2], r[p2:p2 + U], r[p2 + U:p2 + 2 * U], r[p2 + 2 * U:], cnt))
        return out
    return outs, results


def _evidence_outputs(ev):
    """pipsort_outputs over the rows of ev [k, 3] (total, noCausal[0], noCausal[1]); every per-SNP member NULL."""
    ev = ev.reshape(-1, 3)
    outs = (_OutputsV * max(len(ev), 1))()
    for i in range(len(ev)):
        b0 = ev[i].ctypes.data
        outs[i] = _OutputsV(b0, None, b0 + 8, None, None, None)
    return outs


def posterior_exhaustive_grid(num_snps, sigma, z, d, K, snp_map, c, priors, device=0, raw_ld=False):
    """One locus, a grid of priors (gamma, p), one exhaustive pass (pipsort_posterior_exhaustive_grid): a list of Results,
    one per prior, each what posterior_exhaustive with that prior returns."""
    num_snps = np.ascontiguousarray(num_snps, dtype=np.int32)
    if isinstance(sigma, (list, tuple)):
        sigma = np.concatenate([np.asarray(s, dtype=np.float64).ravel() for s in sigma])
    if isinstance(z, (list, tuple)):
        z = np.concatenate([np.asarray(v, dtype=np.float64).ravel() for v in z])
    sigma = np.ascontiguousarray(sigma, dtype=np.float64).ravel()
    z = np.ascontiguousarray(z, dtype=np.float64).ravel()
    d = np.ascontiguousarray(d, dtype=np.float64)
    smap = np.ascontiguousarray(snp_map, dtype=np.int32)
    S, U, N = len(num_snps), int(smap.shape[1]), int(num_snps.sum())
    gam, p = _prior_arrays(priors)
    own = (float(gam[0]), float(p[0])) if len(gam) else (0.01, 0.75)     # the locus's own prior: validated, not reported
    loc = _LocusV(S, num_snps.ctypes.data, sigma.ctypes.data, z.ctypes.data, d.ctypes.data, float(K), U, smap.ctypes.data,
                  own[0], own[1], int(c))
    outs, res = _grid_outputs(len(gam), N, S, U)
    cnt = C.c_uint64()
    _check(lib().pipsort_posterior_exhaustive_grid(C.byref(loc), int(device), RAW_LD if raw_ld else 0, int(c), len(gam), _dp(gam),
                                                   _dp(p), outs, C.byref(cnt)))
    return res(int(cnt.value))


_LOCUS_DT = np.dtype([("num_studies", "<i4"), ("num_snps", "<u8"), ("sigma", "<u8"), ("z", "<u8"), ("d", "<u8"), ("K", "<f8"),
                      ("union_count", "<i4"), ("snp_map", "<u8"), ("gamma", "<f8"), ("sharing_param", "<f8"),
                      ("max_causal", "<i4")], align=True)            # == struct pipsort_locus (checked against ctypes below)
_OUT_DT = np.dtype([(n, "<u8") for n in ("total", "postValues", "noCausal", "sharedPips", "sharedLL", "notSharedLL")])
assert _LOCUS_DT.itemsize == C.sizeof(_LocusV) and _OUT_DT.itemsize == C.sizeof(_OutputsV)
assert all(_LOCUS_DT.fields[n][1] == getattr(_LocusV, n).offset for n, _ in _LocusV._fields_)


def _ready(a, dtype):
    """a as a C-contiguous array of dtype (no copy when it already is one)."""
    if type(a) is np.ndarray and a.dtype == dtype and a.flags.c_contiguous:
        return a
    return np.ascontiguousarray(a, dtype=dtype)


class LocusBatch:
    """The argument block of pipsort_posterior_exhaustive_batch, built once: arrays of `pipsort_locus` / `pipsort_outputs`
    structs (numpy structured arrays filled column by column) that point into the caller's host arrays, and ONE result
    buffer for all loci.  run() is the C-ABI call and nothing else; results() slices the buffer into Results.
    loci: sequence of dicts with the keys of posterior_exhaustive's arguments (num_snps, sigma, z, d, K, snp_map and
    optionally gamma, sharing_param); sigma / z flat float64 arrays (studies concatenated).
    priors: a list of (gamma, p) -- run() is then pipsort_posterior_exhaustive_grid_batch, one result block per locus and
    prior (results() gives a list of Results per locus); evidence_only=True leaves every per-SNP member NULL (the evidence
    read) and the buffer holds (total, noCausal[0], noCausal[1]) per locus and prior, read with evidence().
    class_evidence=True: run() is pipsort_class_evidence_batch, the buffer holds every locus's class table
    ((c+1)(c+2)/2 doubles, Engine.read_class_evidence's layout), read with tables().
    count_table=True: run() is pipsort_count_table_batch, the buffer holds every locus's count table (C(c+3, 3) doubles,
    Engine.read_count_table's layout), read with tables().
    search=True: run() is pipsort_sss_batch, the shotgun search of every locus at max_causal c with at most max_iterations
    rounds; results() as for the ordinary batch, and the arrays `iterations` and `stop_reasons` hold what Engine.sss returns
    with them."""

    def __init__(self, loci, c, device=0, raw_ld=False, priors=None, evidence_only=False, class_evidence=False,
                 count_table=False, search=False, max_iterations=1000):
        if evidence_only and priors is None:
            raise ValueError("evidence_only needs priors")
        if (class_evidence or count_table) and priors is not None:
            raise ValueError("class_evidence and count_table take no priors")
        if class_evidence and count_table:
            raise ValueError("one table read per batch: class_evidence or count_table")
        if search and (priors is not None or class_evidence or count_table):
            raise ValueError("a search batch takes no priors and reads no tables")
        n = self.n = len(loci)
        self.c, self.device, self.flags = int(c), int(device), RAW_LD if raw_ld else 0
        f64, i32 = np.dtype(np.float64), np.dtype(np.int32)
        ns = [_ready(Lc["num_snps"], i32) for Lc in loci]
        sg = [_ready(Lc["sigma"], f64) for Lc in loci]
        zz = [_ready(Lc["z"], f64) for Lc in loci]
        dd = [_ready(Lc["d"], f64) for Lc in loci]
        sm = [_ready(Lc["snp_map"], i32) for Lc in loci]
        self._keep = (ns, sg, zz, dd, sm)                    # the structs hold raw pointers into these
        ptr = lambda arrs: [a.ctypes.data for a in arrs]     # noqa: E731
        S = self.S = np.fromiter((a.shape[0] for a in ns), dtype=np.int64, count=n)
        U = self.U = np.fromiter((a.shape[1] for a in sm), dtype=np.int64, count=n)
        N = self.N = np.fromiter((sum(a.tolist()) for a in ns), dtype=np.int64, count=n)
        la = self.la = np.zeros(n, dtype=_LOCUS_DT)
        la["num_studies"] = S
        la["num_snps"] = ptr(ns); la["sigma"] = ptr(sg); la["z"] = ptr(zz); la["d"] = ptr(dd); la["snp_map"] = ptr(sm)
        la["K"] = [Lc["K"] for Lc in loci]
        la["union_count"] = U
        la["gamma"] = [Lc.get("gamma", 0.01) for Lc in loci]
        la["sharing_param"] = [Lc.get("sharing_param", 0.75) for Lc in loci]
        la["max_causal"] = self.c
        self.priors = None if priors is None else _prior_arrays(priors)
        self.evidence_only = bool(evidence_only)
        self.class_evidence = bool(class_evidence)
        self.count_table = bool(count_table)
        self.search = bool(search)
        self.ntab = _ncnt(self.c) if count_table else _ntab(self.c)
        k = self.k = 1 if priors is None else len(self.priors[0])      # result blocks per locus: locus i, prior j -> i * k + j
        if class_evidence or count_table:
            buf = self.buf = np.empty(n * self.ntab)
            oa = self.oa = np.zeros(0, dtype=_OUT_DT)
        elif evidence_only:
            buf = self.buf = np.empty(n * k * 3)
            b0 = buf.ctypes.data + 24 * np.arange(n * k, dtype=np.int64)
            oa = self.oa = np.zeros(n * k, dtype=_OUT_DT)              # per-SNP members NULL
            oa["total"] = b0
            oa["noCausal"] = b0 + 8
        else:
            # one result buffer: per block total | postValues[N] | noCausal[S] | sharedPips[U] | sharedLL[U] | notSharedLL[U]
            Nb, Sb, Ub = np.repeat(N, k), np.repeat(S, k), np.repeat(U, k)
            off = self.off = np.zeros(n * k + 1, dtype=np.int64)
            np.cumsum(1 + Nb + Sb + 3 * Ub, out=off[1:])
            buf = self.buf = np.empty(int(off[-1]))
            b0 = buf.ctypes.data + 8 * off[:-1]
            oa = self.oa = np.zeros(n * k, dtype=_OUT_DT)
            oa["total"] = b0
            oa["postValues"] = b0 + 8
            oa["noCausal"] = b0 + 8 * (1 + Nb)
            oa["sharedPips"] = b0 + 8 * (1 + Nb + Sb)
            oa["sharedLL"] = b0 + 8 * (1 + Nb + Sb + Ub)
            oa["notSharedLL"] = b0 + 8 * (1 + Nb + Sb + 2 * Ub)
        self.cnt = np.zeros(n, dtype=np.uint64)
        lp, op = C.cast(la.ctypes.data, C.POINTER(_LocusV)), C.cast(oa.ctypes.data, C.POINTER(_OutputsV))
        cp = C.cast(self.cnt.ctypes.data, C.POINTER(C.c_uint64))
        if search:
            self.iterations = np.zeros(n, dtype=np.int32)
            self.stop_reasons = np.zeros(n, dtype=np.int32)
            i32p = C.POINTER(C.c_int32)
            self._args = (lp, n, self.device, self.flags, self.c, int(max_iterations), op,
                          C.cast(self.iterations.ctypes.data, i32p), C.cast(self.stop_reasons.ctypes.data, i32p), cp)
        elif class_evidence or count_table:
            self._args = (lp, n, self.device, self.flags, self.c, _dp(buf), cp)
        elif priors is None:
            self._args = (lp, n, self.device, self.flags, self.c, op, cp)
        else:
            gam, p = self.priors
            self._args = (lp, n, self.device, self.flags, self.c, k, _dp(gam), _dp(p), op, cp)

    def run(self):
        """pipsort_posterior_exhaustive_batch (pipsort_posterior_exhaustive_grid_batch with priors): host buffers in, host
        buffers out."""
        if self.search:                     # the arguments are checked even for an empty list
            _check(lib().pipsort_sss_batch(*self._args))
        elif self.class_evidence:
            _check(lib().pipsort_class_evidence_batch(*self._args))
        elif self.count_table:
            _check(lib().pipsort_count_table_batch(*self._args))
        elif self.priors is not None:       # the priors are validated even for an empty list
            _check(lib().pipsort_posterior_exhaustive_grid_batch(*self._args))
        elif self.n:
            _check(lib().pipsort_posterior_exhaustive_batch(*self._args))
        return self

    def results(self):
        """A Results per locus; with priors, a list of Results (one per prior) per locus."""
        if self.evidence_only or self.class_evidence or self.count_table:
            raise ValueError("an evidence-only or table batch has no per-SNP results: use evidence() / tables()")
        out, buf, k = [], self.buf, self.k
        offl, Nl, Sl, Ul, cl = self.off.tolist(), self.N.tolist(), self.S.tolist(), self.U.tolist(), self.cnt.tolist()
        for i in range(self.n):
            blocks = []
            for o in offl[i * k:(i + 1) * k]:
                Ni, Si, Ui = Nl[i], Sl[i], Ul[i]
                p1 = o + 1 + Ni
                p2 = p1 + Si
                blocks.append(Results(float(buf[o]), buf[o + 1:p1], buf[p1:p2], buf[p2:p2 + Ui], buf[p2 + Ui:p2 + 2 * Ui],
                                      buf[p2 + 2 * Ui:p2 + 3 * Ui], cl[i]))
            out.append(blocks if self.priors is not None else blocks[0])
        return out

    def evidence(self):
        """ndarray [n_loci, n_priors, 3] of (total, noCausal[0], noCausal[1]) (a batch with priors)."""
        if self.priors is None:
            raise ValueError("evidence() needs a batch with priors")
        if self.evidence_only:
            return self.buf.reshape(self.n, self.k, 3).copy()
        o = self.off[:-1]
        nc = o + 1 + np.repeat(self.N, self.k)
        return np.stack([self.buf[o], self.buf[nc], self.buf[nc + 1]], axis=-1).reshape(self.n, self.k, 3)

    def tables(self):
        """ndarray [n_loci, (c+1)(c+2)/2] of class tables (a class_evidence batch) or [n_loci, C(c+3, 3)] of count tables
        (a count_table batch)."""
        if not (self.class_evidence or self.count_table):
            raise ValueError("tables() needs a class_evidence or count_table batch")
        return self.buf.reshape(self.n, self.ntab).copy()


def posterior_exhaustive_batch(loci, c, device=0, raw_ld=False):
    """A list of loci in one call (pipsort_posterior_exhaustive_batch): the engine pipelines them over three streams, so
    the uploads / preparation of the next locus and the read-back of the previous one overlap the current evaluation.
    Returns a list of Results.  (LocusBatch separates building the argument block from the call itself.)"""
    return LocusBatch(loci, c, device, raw_ld).run().results()


def posterior_exhaustive_grid_batch(loci, c, priors, device=0, raw_ld=False, evidence_only=False):
    """A grid of priors (gamma, p) for a list of loci in one call (pipsort_posterior_exhaustive_grid_batch): one exhaustive
    pass per locus, pipelined as posterior_exhaustive_batch.  Returns a list (per locus) of lists (per prior) of Results,
    or with evidence_only=True the ndarray [n_loci, n_priors, 3] of (total, noCausal[0], noCausal[1])."""
    B = LocusBatch(loci, c, device, raw_ld, priors=priors, evidence_only=evidence_only).run()
    return B.evidence() if evidence_only else B.results()


def class_evidence_batch(loci, c, device=0, raw_ld=False):
    """The class table of every locus (pipsort_class_evidence_batch): one class-resolved pass per locus, pipelined as
    posterior_exhaustive_batch.  loci as posterior_exhaustive_batch takes them; returns ndarray [n_loci, (c+1)(c+2)/2]."""
    return LocusBatch(loci, c, device, raw_ld, class_evidence=True).run().tables()


def count_table_batch(loci, c, device=0, raw_ld=False):
    """The count table of every locus (pipsort_count_table_batch): one pass per locus on a store with the count table,
    pipelined as posterior_exhaustive_batch.  loci as posterior_exhaustive_batch takes them; returns ndarray
    [n_loci, C(c+3, 3)] (Engine.read_count_table's layout)."""
    return LocusBatch(loci, c, device, raw_ld, count_table=True).run().tables()


def sss_batch(loci, c, max_iterations=1000, device=0, raw_ld=False):
    """The shotgun search of every locus (pipsort_sss_batch): what Engine.sss(c, max_iterations) returns on a fresh engine
    per locus, with several searches in flight per host thread.  loci as posterior_exhaustive_batch takes them.  Returns
    (a list of Results, iterations, stop_reasons), the last two int32 ndarrays with one entry per locus (stop reason 0 =
    iteration cap, 1 = no new configuration, 2 = convergence)."""
    B = LocusBatch(loci, c, device, raw_ld, search=True, max_iterations=max_iterations).run()
    return B.results(), B.iterations.copy(), B.stop_reasons.copy()


def _count_c(w):
    c = next((k for k in range(KMAX + 1) if _ncnt(k) == w), -1)
    if c < 0:
        raise ValueError(f"a count table has C(c+3, 3) entries for some c in [0, {KMAX}], not {w}")
    return c


def count_posterior(tables, union_counts, gamma, p):
    """The posterior of the numbers of causal SNPs under the prior (gamma, p), per locus (pipsort_count_posterior, host
    code, no device).  tables: [n_loci, C(c+3, 3)] from count_table_batch or Engine.read_count_table; union_counts: U per
    locus.  Returns (post, log_evidence): post[i, a, b0, b1] is the posterior probability that locus i has a SNPs causal in
    both studies, b0 in study 0 only and b1 in study 1 only (zero outside a + b0 + b1 <= c), an ndarray of shape
    (n, c+1, c+1, c+1); log_evidence[i] is the locus's log evidence at that prior (the grid read's total).  The marginals:
      P(a >= 1)  = 1 - post[i, 0].sum()                     -- at least one causal SNP shared by the two studies;
      P(k0 = n)  = sum over a + b0 = n of post[i, a, b0, :]  -- n causal SNPs in study 0 (k0 = a + b0);
      P(k1 = n)  = sum over a + b1 = n of post[i, a, :, b1]  -- the same for study 1 (k1 = a + b1)."""
    tab = np.ascontiguousarray(tables, dtype=np.float64)
    if tab.ndim != 2:
        raise ValueError("tables must be [n_loci, C(c+3, 3)]")
    n, w = tab.shape
    c = _count_c(w)
    U = np.ascontiguousarray(union_counts, dtype=np.int32).ravel()
    if U.size != n:
        raise ValueError("one union count per locus")
    flat, ev = np.empty((n, w)), np.empty(n)
    _check(lib().pipsort_count_posterior(n, c, _dp(tab), U.ctypes.data_as(C.POINTER(C.c_int32)), float(gamma), float(p),
                                         _dp(flat), _dp(ev)))
    post = np.zeros((n, c + 1, c + 1, c + 1))
    cls = np.array(_cnt_classes(c))
    post[:, cls[:, 1], cls[:, 2], cls[:, 3]] = flat
    return post, ev


def class_tables_from_counts(tables, c=None):
    """Class tables ([n_loci, (c+1)(c+2)/2], Engine.read_class_evidence's layout) from count tables ([n_loci, C(c+3, 3)]): a
    log-sum-exp over b0 per class (J, a), so that one count_table_batch also feeds fit_prior.  c (optional) must match the
    tables' width."""
    tab = np.asarray(tables, dtype=np.float64)
    one = tab.ndim == 1
    tab = tab.reshape(1, -1) if one else tab
    cw = _count_c(tab.shape[1])
    if c is not None and int(c) != cw:
        raise ValueError(f"count tables of width {tab.shape[1]} are for c={cw}, not {c}")
    out = np.empty((tab.shape[0], _ntab(cw)))
    k = 0
    for J in range(cw + 1):
        for a in range(J + 1):
            part = tab[:, k:k + J - a + 1]
            m = part.max(axis=1)
            safe = np.where(np.isneginf(m), 0.0, m)
            with np.errstate(divide="ignore"):
                out[:, J * (J + 1) // 2 + a] = np.where(np.isneginf(m), -np.inf,
                                                        safe + np.log(np.exp(part - safe[:, None]).sum(axis=1)))
            k += J - a + 1
    return out[0] if one else out


_FIT = {"gamma": 1, "p": 2, "gamma,p": 3}


def fit_prior(tables, union_counts, fit="p", gamma=0.01, p=0.75):
    """The prior of largest joint log evidence over the loci of `tables` ([n_loci, (c+1)(c+2)/2], from class_evidence_batch
    or Engine.read_class_evidence; union_counts: U per locus) -- pipsort_fit_prior, host code, no device.  fit: "p",
    "gamma", "gamma,p", or the bit mask itself (1 gamma, 2 p; 0 evaluates at (gamma, p) only); a parameter not fitted keeps
    the value given.  Returns (gamma, p, joint_log_evidence, per_locus_log_evidence).  Then run posterior_exhaustive_batch at
    that prior for the PIPs."""
    if isinstance(fit, str) and fit not in _FIT:
        raise ValueError(f"fit must be one of {sorted(_FIT)} or a bit mask")
    bits = _FIT[fit] if isinstance(fit, str) else int(fit)
    tab = np.ascontiguousarray(tables, dtype=np.float64)
    if tab.ndim != 2:
        raise ValueError("tables must be [n_loci, (c+1)(c+2)/2]")
    n, w = tab.shape
    c = next((k for k in range(KMAX + 1) if _ntab(k) == w), -1)
    if c < 0:
        raise ValueError(f"a class table has (c+1)(c+2)/2 entries for some c in [0, {KMAX}], not {w}")
    U = np.ascontiguousarray(union_counts, dtype=np.int32).ravel()
    if U.size != n:
        raise ValueError("one union count per locus")
    g, q, joint = C.c_double(gamma), C.c_double(p), C.c_double()
    per = np.empty(n)
    _check(lib().pipsort_fit_prior(n, c, _dp(tab), U.ctypes.data_as(C.POINTER(C.c_int32)), bits, C.byref(g), C.byref(q),
                                   C.byref(joint), _dp(per)))
    return g.value, q.value, joint.value, per


def preprocess_study(ld, z, device=0):
    """Model's per-study pre-processing (model.h:171-264) on the GPU: returns (sigma_eff, info dict)."""
    ld = np.ascontiguousarray(ld, dtype=np.float64)
    z = np.ascontiguousarray(z, dtype=np.float64)
    n = ld.shape[0]
    assert ld.shape == (n, n) and z.shape == (n,)
    out = np.empty((n, n))
    info = _PrepInfo()
    _check(lib().pipsort_preprocess_study(int(device), n, _dp(ld), _dp(z), _dp(out), C.byref(info)))
    return out, {k: getattr(info, k) for k, _ in _PrepInfo._fields_}


def shard_ranks_for_map(snp_map, c, parts, keep_order=False):
    """pipsort_shard_ranks without an engine (pure host arithmetic, no device needed)."""
    smap = np.ascontiguousarray(snp_map, dtype=np.int32)
    b = (C.c_uint64 * (parts + 1))()
    _check(lib().pipsort_shard_ranks_for_map(smap.ctypes.data_as(C.POINTER(C.c_int32)), int(smap.shape[1]), int(c),
                                             int(parts), KEEP_ORDER if keep_order else 0, b))
    return [int(x) for x in b]


def measure_fp64_peak(device=0):
    out = C.c_double()
    _check(lib().pipsort_measure_fp64_peak(int(device), C.byref(out)))
    return float(out.value)


def version():
    return lib().pipsort_version().decode()
