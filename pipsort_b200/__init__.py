"""pipsort_b200: B200-native (sm_100a) posterior-calculation engine behind PIPSORT's PostCal boundary."""
from .engine import (Engine, PipsortError, Results, measure_fp64_peak, posterior_exhaustive, posterior_exhaustive_batch, posterior_exhaustive_grid, posterior_exhaustive_grid_batch, LocusBatch, preprocess_study, shard_ranks_for_map, version, lib,  # noqa: F401
                     KEEP_ORDER, KMAX, PRIOR_CLASSES)
