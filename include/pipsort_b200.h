/* pipsort_b200 -- C-ABI of the B200 (sm_100a) posterior-calculation engine.
 *
 * This is the drop-in boundary for PIPSORT's PostCal hot path (SURVEY.md section 8b).  Every entry
 * point cites the reference interface it replaces (paths relative to the PIPSORT source tree).
 * Plain C types only; no torch, no C++ types.  All functions return 0 on success and a non-zero
 * PIPSORT_E_* code on failure; pipsort_last_error() returns a human-readable message for the last
 * failure on the calling thread.  The engine is single-caller (like PostCal, which is driven from
 * the main thread after omp_set_num_threads(1), pipsort.cpp:222) and never retains host pointers:
 * inputs are copied to the device in pipsort_create, outputs are written into caller-owned buffers.
 *
 * There is NO CPU fallback: every compute entry point fails with PIPSORT_E_CUDA when no CUDA device
 * is usable.
 */
#ifndef PIPSORT_B200_H
#define PIPSORT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIPSORT_OK 0
#define PIPSORT_E_ARG 1      /* bad argument (message says which)                                  */
#define PIPSORT_E_CUDA 2     /* CUDA runtime failure / no device                                   */
#define PIPSORT_E_STUDIES 3  /* number of studies != 2 (postcal.cpp:20-23 exits for > 2)           */
#define PIPSORT_E_RANGE 4    /* rank space / exponent range overflow                               */
#define PIPSORT_E_SINGULAR 5 /* a causal sub-block lost positive definiteness (postcal.cpp:291-294) */
#define PIPSORT_E_CONFIG 6   /* an explicit configuration row the reference aborts on (postcal.cpp:593-596) */

#define PIPSORT_KMAX 8       /* max union SNPs per configuration on the scoring path               */
#define PIPSORT_JMAX_EXH 3   /* exhaustive path: union subsets of size <= 3 (postcal.cpp:760-762)  */

/* pipsort_create flags */
#define PIPSORT_KEEP_ORDER 1u /* keep the snp_map order internally (default: union SNPs are relabelled
                                 by type so that warps run one code path; sums are order independent) */

#define PIPSORT_GENERIC_ONLY 2u /* testing: run every subset-size class through the generic (warp per configuration)
                                  kernel instead of the register kernel                                */

#define PIPSORT_RAW_LD 4u     /* pipsort_locus.sigma holds the LD matrices as read from the -l files and K is ignored: the engine
                                 runs Model's pre-processing (PSD shift + eigen-decomposition, model.h:171-264) on the device */

#define PIPSORT_PRIOR_CLASSES 8u /* class-resolved store: the accumulators are kept unweighted per prior class (subset size J,
                                   number a of SNPs causal in both studies), so that one exhaustive pass serves any number of
                                   priors (gamma, p) -- pipsort_read_prior_grid.  The locus's gamma / sharing_param stay the
                                   engine's own prior: pipsort_read_accumulators, pipsort_finalize(_reset) and pipsort_fetch_results
                                   report it.  Such an engine refuses pipsort_sss(_sharded), pipsort_score_union_configs*,
                                   pipsort_score_given_configs* and pipsort_p2p_combine_finalize (PIPSORT_E_ARG). */

typedef struct pipsort_engine pipsort_engine;

/* Locus description = the PostCal constructor arguments the likelihood actually consumes
 * (postcal.h:118-195).  The caller (Model, model.h:171-264) has already applied the PSD fix and the
 * eigen-decomposition; what crosses the boundary is, per study s,
 *   sigma_s = B_s^T B_s  (the effective LD; B = |Omega|^(1/2) Q^T is PostCal's BIG_SIGMA block), n_s x n_s,
 *             row-major (symmetric, so arma's column-major is the same bytes), studies concatenated;
 *   z_s     = B_s^T S'_s (S' is PostCal's S_LONG_VEC), n_s doubles, studies concatenated;
 *   d_s     = s_squared * n_s / min(n) + t_squared   (postcal.cpp:66,89; only the diagonal of sigmaC
 *             reaches the likelihood, postcal.cpp:250);
 *   K       = S'^T S'  (postcal.cpp:285-287 with an empty causal set);
 *   snp_map = PostCal::idx_to_snp_map, int32[S][U], study index of union SNP g or -1 (model.h:132).
 */
typedef struct pipsort_locus {
    int32_t num_studies;       /* S, must be 2                                                     */
    const int32_t* num_snps;   /* [S]      PostCal::num_snps_all                                   */
    const double* sigma;       /* [sum n_s^2]                                                      */
    const double* z;           /* [sum n_s]                                                        */
    const double* d;           /* [S]                                                              */
    double K;
    int32_t union_count;       /* U        PostCal::unionSnpCount                                  */
    const int32_t* snp_map;    /* [S*U]                                                            */
    double gamma;              /* PostCal::gamma                                                   */
    double sharing_param;      /* PostCal::sharing_param (p)                                       */
    int32_t max_causal;        /* PostCal::maxCausalSNP (c); sizes the exponent range              */
} pipsort_locus;

/* Caller-owned output block = PostCal's result members (postcal.h:62-99), all in log space with 0.0
 * meaning "nothing accumulated" exactly as addlogSpace leaves them (postcal.h:102-112).           */
typedef struct pipsort_outputs {
    double* total;        /* [1]   totalLikeLihoodLOG / sss_sum_lkl                                 */
    double* postValues;   /* [N]   N = sum n_s, indexed offset_s + i  (postcal.cpp:1020-1030)        */
    double* noCausal;     /* [S]   (postcal.cpp:988-1000)                                           */
    double* sharedPips;   /* [U]   (postcal.cpp:1003-1012)                                          */
    double* sharedLL;     /* [U]                                                                    */
    double* notSharedLL;  /* [U]   (postcal.cpp:1014-1016)                                          */
} pipsort_outputs;

/* Replaces Model's per-study pre-processing (model.h:171-264): makeSigmaPositiveSemiDefinite (util.cpp:195-226: +0.01
 * on the diagonal until the LU determinant is > 0, an underflowed determinant counting as not positive), eigen_decomp
 * (util.cpp:228-263), |Omega| (model.h:227), B = |Omega|^(1/2) Q^T and S' = |Omega|^(-1/2) Q^T z (model.h:230-255) --
 * returned in the form the engine consumes: sigma_eff = B^T B (n x n, host), K = S'^T S', plus the diagonal shift.
 * Runs on `device` (cuSOLVER LU / symmetric eigensolver + the engine's own kernels); host buffers in and out.
 * pipsort_create with PIPSORT_RAW_LD does the same without the round trip through host memory; its findings are read
 * back with pipsort_prep_info_get.                                                                   */
typedef struct pipsort_prep_info {
    double add_diag;        /* a_s: what makeSigmaPositiveSemiDefinite added to the diagonal                      */
    double K;               /* S'_s^T S'_s                                                                        */
    double min_abs_eig;     /* smallest |eigenvalue| of the shifted matrix                                        */
    int32_t n_negative;     /* eigenvalues whose sign model.h:227 flips                                           */
    int32_t psd_iterations; /* LU factorizations the PSD loop needed                                              */
} pipsort_prep_info;
int pipsort_preprocess_study(int device, int32_t n, const double* ld, const double* z, double* sigma_eff,
                             pipsort_prep_info* info);
int pipsort_prep_info_get(const pipsort_engine* e, int study, pipsort_prep_info* info);

/* Replaces the PostCal constructor (postcal.h:118-195): copies the locus to `device` (CUDA ordinal),
 * builds the device-side tables and zeroes the accumulators.                                       */
int pipsort_create(const pipsort_locus* locus, int device, uint32_t flags, pipsort_engine** out);

/* Replaces PostCal::~PostCal (postcal.h:197-204). */
void pipsort_destroy(pipsort_engine* e);

/* Zero the accumulators (a fresh PostCal has all-zero result arrays, postcal.h:129-160). */
int pipsort_reset(pipsort_engine* e);

/* Number of union subsets of size 0..c = the reference's total_iteration (postcal.cpp:723-725). */
int pipsort_total_ranks(const pipsort_engine* e, int c, uint64_t* out);

/* Replaces PostCal::computeTotalLikelihood (postcal.cpp:716-1092) restricted to the union-subset
 * ranks [rank_begin, rank_end) in the reference's size-then-lexicographic order (nextBinary /
 * findConfig, postcal.cpp:307-387) over the engine's SNP order (= the snp_map order when the engine
 * was created with PIPSORT_KEEP_ORDER; a fixed relabelling of it otherwise, so a partition of
 * [0,total) always reproduces the whole run).  Accumulates into the engine's device accumulators
 * (asynchronously on the engine's stream); n_configs (optional) receives the number of expanded
 * configurations evaluated so far after a stream sync.                                            */
int pipsort_run_exhaustive(pipsort_engine* e, int c, uint64_t rank_begin, uint64_t rank_end);

/* Replaces the body of the OpenMP loop of sss_computeTotalLikelihood, i.e. a batch of
 * expand_and_compute_lkl calls (sss_postcal.cpp:223-255, 447-685): idx is int32[n][kmax] of union
 * indices in snp_map order, -1 padded; make_updates (uint8[n], NULL = all 1) says which
 * configurations are added to the accumulators; out_max_abs_l[n] receives the expansion value with
 * the largest |l| (sss_postcal.cpp:560,624-626; 0.0 when no expansion exists).  Host buffers.       */
int pipsort_score_union_configs(pipsort_engine* e, const int32_t* idx, int64_t n, int kmax,
                                const uint8_t* make_updates, double* out_max_abs_l);

/* Same with device-resident idx / make_updates / out buffers (no host copies, asynchronous). */
int pipsort_score_union_configs_device(pipsort_engine* e, const int32_t* d_idx, int64_t n, int kmax,
                                       const uint8_t* d_make_updates, double* d_out_max_abs_l);

/* (The exponent range of the accumulators is sized from pipsort_locus.max_causal: create the engine with max_causal >= the
 * largest number of causal SNPs a row may hold -- PIPSORT_KMAX covers every row this call accepts; the reference does not
 * bound a row by maxCausalSNP.)
 * Replaces PostCal::computeTotalLikelihoodGivenConfigs (postcal.cpp:400-714; flags -b/-d/-e, pipsort.cpp:153-161):
 * configs is the int16 matrix [num_configs][num_groups] the reference mmaps (postcal.cpp:429-447), every row ONE
 * configuration given as global SNP indices offset_s + i (postcal.cpp:868-872) in increasing order, negative =
 * unused group; rows without any entry are the null configuration (postcal.cpp:461-492).  Accumulates into the
 * engine's accumulators (read them with pipsort_read_accumulators; pipsort_config_count gives the reference's
 * mycount).  A row the reference aborts on ("This did not work as expected", postcal.cpp:593-596: entries out of
 * order or repeated), an entry >= N, or more than PIPSORT_KMAX causal SNPs in one study fails with
 * PIPSORT_E_CONFIG (reported by this call for host buffers, by the next pipsort_read_accumulators for the
 * asynchronous device-buffer variant).                                                             */
int pipsort_score_given_configs(pipsort_engine* e, const int16_t* configs, int64_t num_configs, int num_groups);
int pipsort_score_given_configs_device(pipsort_engine* e, const int16_t* d_configs, int64_t num_configs, int num_groups);

/* Replaces PostCal::sss_computeTotalLikelihood (sss_postcal.cpp:102-380): the whole stochastic shotgun search from the
 * empty configuration -- std::mt19937(12345), at most max_iterations (the reference: 1000) rounds of
 * zero ++ minus ++ plus neighbourhoods (sss_postcal.cpp:20-99), every unseen neighbour expanded + scored +
 * accumulated in ONE launch, the three within-group std::discrete_distribution draws and the draw across groups
 * (sss_postcal.cpp:289-343), the "no new configuration" break (:260-263) and the 1e-3 convergence rule after 100
 * rounds (:265-270).  The explored-configuration map (PostCal::config_hashmap, postcal.h:98) is a hash table in device
 * memory; per round only the current configuration goes to the device and the neighbours' values come back.
 * Accumulates into the engine's accumulators (call pipsort_reset first for a fresh PostCal); *iterations receives the
 * number of completed rounds, *stop_reason 0 = max_iterations reached, 1 = break condition, 2 = convergence.     */
int pipsort_sss(pipsort_engine* e, int max_causal, int max_iterations, int32_t* iterations, int32_t* stop_reason);
/* The same search with every round's neighbourhood split over the GPUs of a group (the loop the reference
 * parallelises with OpenMP, sss_postcal.cpp:223-255).  One process per GPU; every rank has created its engine from the
 * same locus and called pipsort_p2p_export / pipsort_p2p_connect; all ranks call this function with the same arguments.
 * Every rank keeps a replica of the explored-configuration table and follows the same trajectory (same seed, same
 * values); of a round's unseen neighbours rank r expands + scores + accumulates those with index r (mod world), the
 * max-|l| values go to every peer through the mailboxes (device-side stores over NVLink, no collective library).  The
 * accumulators stay RANK-PARTIAL: combine them afterwards (pipsort_p2p_reduce_to_root, then read on the root).        */
int pipsort_sss_sharded(pipsort_engine* e, int max_causal, int max_iterations, int32_t* iterations, int32_t* stop_reason);
/* Forget the explored configurations (pipsort_sss does this itself when it starts). */
int pipsort_sss_reset(pipsort_engine* e);

/* Reads the accumulators into PostCal's result arrays (any member of `out` may be NULL).  Replaces the
 * reads of totalLikeLihoodLOG / postValues / noCausal / sharedPips / sharedLL / notSharedLL by
 * findOptimalSetGreedy (postcal.cpp:1144-1163) and printPost2File (postcal.h:288-336).            */
int pipsort_read_accumulators(pipsort_engine* e, const pipsort_outputs* out);

/* Launches the finalize kernel only (bins -> log-space results, kept on the device); pipsort_read_accumulators
 * = pipsort_finalize + device-to-host copy + scatter into the caller's arrays.                      */
int pipsort_finalize(pipsort_engine* e);

/* pipsort_finalize that also leaves the accumulators EMPTY (the same launch zeroes every bin it has read and the
 * counters): a driver that repeats passes -- permutation replicates, one locus after another on a resident engine --
 * needs no pipsort_reset between them.  The results stay on the device until the next finalize;
 * pipsort_fetch_results copies them into the caller's arrays (same layout and meaning as pipsort_read_accumulators,
 * which would find the store empty after a pipsort_finalize_reset).  Replaces the zero-initialised result arrays of a
 * fresh PostCal (postcal.h:129-160) + the reads of postcal.cpp:1144-1163.                            */
int pipsort_finalize_reset(pipsort_engine* e);
int pipsort_fetch_results(pipsort_engine* e, const pipsort_outputs* out);

/* Device time (CUDA events on the engine's stream) of the dominant kernel of the last pipsort_run_exhaustive
 * call: the launch that covered the largest subset-size class.  Blocks until that launch has finished. */
int pipsort_last_kernel_ms(pipsort_engine* e, float* ms);

/* Number of expanded configurations accumulated since the last reset (the reference's mycount). */
int pipsort_config_count(pipsort_engine* e, uint64_t* out);

/* One locus, one call: what Model::run does with a fresh PostCal (model.h:265-276: new PostCal, findOptimalSetGreedy ->
 * computeTotalLikelihood, read the result members) -- pipsort_create + pipsort_run_exhaustive over the whole rank space +
 * pipsort_read_accumulators + pipsort_destroy.  Host buffers in (locus), host buffers out (out); n_configs (optional)
 * receives the reference's mycount.                                                                    */
int pipsort_posterior_exhaustive(const pipsort_locus* locus, int device, uint32_t flags, int c, const pipsort_outputs* out,
                                 uint64_t* n_configs);

/* Results for a grid of priors from ONE pass (engine created with PIPSORT_PRIOR_CLASSES): outs[i] receives what an engine
 * created with gamma[i] / sharing_param[i] would report after the same calls -- same layout and meaning as
 * pipsort_read_accumulators (0.0 = nothing accumulated with a non-zero prior weight); n_configs (optional) the configuration
 * count, the same for every prior.  The likelihood E_0(C0) E_1(C1) of an expanded configuration does not depend on the prior,
 * and the prior pi'(J,a) (postcal.cpp:19-59) only on the subset size J and the number a of SNPs causal in both studies, so the
 * store keeps one unweighted sum per (SNP, J, state, a') and per (J, a) and the weights are applied here: one finalize launch
 * over all priors and one device-to-host copy.  Every prior is validated as pipsort_create does (gamma in (0,1), p in [0,1]);
 * n_priors >= 1.  The store may be the sum of several engines' (pipsort_merge, an all-reduce of pipsort_accumulator_buffer,
 * pipsort_p2p_reduce_to_root).  When every block leaves postValues, sharedPips, sharedLL and notSharedLL NULL, only total and
 * noCausal are formed and copied back (an evidence read: the same values, bit for bit, at a fraction of the cost).       */
int pipsort_read_prior_grid(pipsort_engine* e, int n_priors, const double* gamma, const double* sharing_param,
                            const pipsort_outputs* outs, uint64_t* n_configs);

/* One locus, a grid of priors, one call: pipsort_create (flags | PIPSORT_PRIOR_CLASSES) + pipsort_run_exhaustive over the whole
 * rank space + pipsort_read_prior_grid + pipsort_destroy.  The locus's own gamma / sharing_param are validated but not reported. */
int pipsort_posterior_exhaustive_grid(const pipsort_locus* locus, int device, uint32_t flags, int c, int n_priors, const double* gamma,
                                      const double* sharing_param, const pipsort_outputs* outs, uint64_t* n_configs);

/* The same for a list of loci (a fine-mapping run has thousands): software pipelines over three engines on three
 * streams each, driven by a few host threads (PIPSORT_BATCH_THREADS, default 3; lists of fewer than 8 loci: one), so that
 * the uploads and preparation launches of the next loci and the read-back of the previous ones overlap the evaluation of
 * the current ones.  loci[i] -> outs[i] (and n_configs[i], optional).  Stops at the first error.                    */
int pipsort_posterior_exhaustive_batch(const pipsort_locus* loci, int32_t n_loci, int device, uint32_t flags, int c,
                                       const pipsort_outputs* outs, uint64_t* n_configs);

/* A grid of priors for a list of loci: pipsort_posterior_exhaustive_grid for every locus, pipelined as
 * pipsort_posterior_exhaustive_batch pipelines the ordinary pass (same flags; PIPSORT_PRIOR_CLASSES is implied).  Locus i and
 * prior j go to outs[i * n_priors + j], n_configs[i] (optional) receives locus i's configuration count.  Every prior is
 * validated once, before any device work (gamma in (0,1), p in [0,1], n_priors >= 1; PIPSORT_E_ARG names a bad prior); each
 * locus's own gamma / sharing_param is validated as pipsort_create does but not reported.  n_loci == 0 returns 0.  Any
 * member of an output block may be NULL.  When a locus's blocks leave postValues, sharedPips, sharedLL and notSharedLL all
 * NULL, its read is an evidence read: the finalize forms total and noCausal only and copies back 3 doubles per prior --
 * the values the full read gives, bit for bit (the scan over p of a sensitivity analysis needs no more; pipsort_read_prior_grid
 * makes the same choice).  Stops at the first error, as pipsort_posterior_exhaustive_batch does.                      */
int pipsort_posterior_exhaustive_grid_batch(const pipsort_locus* loci, int32_t n_loci, int device, uint32_t flags, int c,
                                            int n_priors, const double* gamma, const double* sharing_param,
                                            const pipsort_outputs* outs, uint64_t* n_configs);

/* The same count as it was when pipsort_read_accumulators last ran (it travels with the results: no extra device
 * round trip).                                                                                     */
int pipsort_last_read_config_count(const pipsort_engine* e, uint64_t* out);

/* Debug / parity: the configuration the reference evaluates at union-subset rank `rank`, expansion
 * number `expansion` (ascending bmask order with checkOR rejects skipped, postcal.cpp:903-958), in
 * snp_map order regardless of the engine's internal relabelling.  out_union_idx[c] gets the chosen
 * union SNPs (ascending, -1 padded), out_state[c] 1 = study 0 only, 2 = study 1 only, 3 = both;
 * *n_expansions the number of accepted expansions of that subset.  Evaluated on the device.        */
int pipsort_enumerate(pipsort_engine* e, int c, uint64_t rank, uint32_t expansion, int32_t* out_union_idx,
                      int32_t* out_state, uint32_t* n_expansions);

/* Multi-GPU: the accumulators are one flat device array of doubles whose element-wise SUM over
 * engines working on disjoint rank ranges of the same locus is the accumulator state of the union
 * (SURVEY.md section 8e); the configuration count and the error counters live in its last elements, so
 * the one sum carries them too.  One process per GPU combines them with a single NCCL all-reduce(sum) on
 * this buffer; a single process driving several devices can use pipsort_merge.                    */
int pipsort_accumulator_buffer(pipsort_engine* e, void** device_ptr, uint64_t* num_doubles);
int pipsort_merge(pipsort_engine* dst, pipsort_engine* src); /* dst += src (copies across devices)  */

/* The same combine step WITHOUT a collective library, over NVLink / NVSwitch peer memory (one process per GPU):
 * every engine exports a mailbox (CUDA IPC handle, PIPSORT_IPC_HANDLE_BYTES bytes; one inbox slot per rank of the
 * group, so the group size is given at export), the launcher exchanges the handles (any side channel:
 * torch.distributed all_gather_object, MPI, a file) and hands every rank the whole table.  After that
 * pipsort_p2p_reduce_to_root -- stream-ordered, asynchronous, called by EVERY rank after its pipsort_run_exhaustive
 * / scoring calls -- makes the non-root ranks copy their accumulator stores straight into their slot of the root's
 * memory (posted 16-byte stores over the link) and makes the root wait (on the device) for all of them and add them
 * to its store: pipsort_read_accumulators on the ROOT then returns the whole job's result.  Engines of one group must
 * be created from the same locus and call in lockstep (the n-th call of every rank belongs together).            */
#define PIPSORT_IPC_HANDLE_BYTES 64
int pipsort_p2p_export(pipsort_engine* e, int world, void* handle);
int pipsort_p2p_connect(pipsort_engine* e, const void* handles, int world, int rank, int root);
int pipsort_p2p_reduce_to_root(pipsort_engine* e);
/* The same, and a NON-root rank's accumulators are left empty by the very kernel that sends them (the root's are emptied
 * by pipsort_finalize_reset): a repeated pass needs no pipsort_reset on any rank.                                 */
int pipsort_p2p_reduce_to_root_reset(pipsort_engine* e);
/* The whole tail of a repeatable multi-GPU pass in ONE launch per rank: a non-root rank sends its store (and empties it); the
 * root sums its own store and the peers' slots straight into the finalize (bins -> results; nothing is written back but
 * zeros) -- the results are then fetched on the root with pipsort_fetch_results.  Stream-ordered, asynchronous.            */
int pipsort_p2p_combine_finalize(pipsort_engine* e);

/* Split [0,total) into `parts` contiguous rank ranges of roughly equal work (expanded configurations
 * weighted); bounds receives parts+1 values.                                                      */
int pipsort_shard_ranks(const pipsort_engine* e, int c, int parts, uint64_t* bounds);
/* The same split computed from the snp_map alone (int32[2][U] as in pipsort_locus; flags as given to pipsort_create):
 * pure host arithmetic, needs no device -- a launcher can plan the shards before any GPU is touched.             */
int pipsort_shard_ranks_for_map(const int32_t* snp_map, int32_t union_count, int c, int parts, uint32_t flags,
                                uint64_t* bounds);

/* Stream the engine works on (cudaStream_t as void*), and a blocking sync on it.  pipsort_set_stream
 * makes the engine issue all further work on a caller-owned stream (e.g. the one a NCCL all-reduce of
 * pipsort_accumulator_buffer is enqueued on); NULL restores the engine's own stream.  The DEFAULT stream is
 * named by cudaStreamLegacy ((void*)1), not by NULL.                                                 */
void* pipsort_stream(pipsort_engine* e);
int pipsort_set_stream(pipsort_engine* e, void* cuda_stream);
int pipsort_sync(pipsort_engine* e);

/* CUDA graphs.  Between pipsort_graph_begin and pipsort_graph_end the engine's asynchronous calls (pipsort_reset,
 * pipsort_run_exhaustive, pipsort_score_*_device, pipsort_p2p_reduce_to_root, pipsort_finalize) are recorded instead of
 * executed; pipsort_graph_launch replays the recorded sequence with ONE launch.  For a locus that takes 0.1 ms the host
 * cost of issuing the half dozen launches of a pass is comparable to the pass itself; a driver that repeats the same
 * pass (bootstrap / permutation replicates, benchmarks) replays the graph.  Run the sequence once normally first (the
 * first pass allocates its scratch buffers), and do not call blocking entry points while capturing.              */
int pipsort_graph_begin(pipsort_engine* e);
int pipsort_graph_end(pipsort_engine* e, int32_t* graph_id);
int pipsort_graph_launch(pipsort_engine* e, int32_t graph_id);

/* Benchmark hygiene: evict L2 by overwriting a scratch buffer larger than L2 on the engine's stream. */
int pipsort_flush_l2(pipsort_engine* e);

/* Device-side timing of the launches issued between begin and end (CUDA events on the engine's
 * stream): milliseconds.                                                                          */
int pipsort_timer_begin(pipsort_engine* e);
int pipsort_timer_end(pipsort_engine* e, float* ms);

/* Number of engine kernels launched since create (bench.py's gpu_launches). */
uint64_t pipsort_launch_count(const pipsort_engine* e);

/* FP64 DFMA micro-benchmark (register-resident FMA chains on every SM): measured FLOP/s of `device`.
 * Used as the roofline denominator (MEASURED_PEAKS.json carries no FP64 figure).                   */
int pipsort_measure_fp64_peak(int device, double* flops_per_sec);

const char* pipsort_last_error(void);
const char* pipsort_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PIPSORT_B200_H */
