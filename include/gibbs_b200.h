/*
 * include/gibbs_b200.h -- C ABI of libgibbs_b200.so, the B200 (sm_100a) replacement for the
 * data-parallel hot path of Etschbeijer/GibbsSampling.
 *
 * Each entry point replaces a piece of /root/reference/GibbsSampling/GibbsSampling.fs (cited as
 * fs:N). The F# module keeps the reference signatures and binds these symbols with P/Invoke
 * (INTEGRATION.md, fsharp/GibbsSamplingB200.fs); in this repository the same symbols are bound
 * with ctypes by gibbssampling_b200/_abi.py.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every host buffer; the library never keeps
 *     a host pointer after a call returns; device memory is owned by the handle
 *   - every function returns a gibbs_status (0 = OK); the text of the last failure is available
 *     from gibbs_last_error(); nothing throws or aborts across the boundary
 *   - sequences: ONE contiguous buffer of upper-case ASCII symbols (BioItem.symbol, fs:17) plus
 *     int64 offsets[n_seqs + 1]. Every symbol the reference's 49-slot tables index ('*'..'Z',
 *     fs:17-20) is accepted, anything else is GIBBS_ERR_SYMBOL. A, C, G, T are the alphabet the
 *     tables are built for; any other symbol is treated as NOT in `alphabet`: its PWM row is 0
 *     (fs:283-287), a window that holds it scores 0, a site base that is one is not counted.
 *     Gap '-' with alphabet_size >= 5 (the script's dnaBases, where Gap IS an alphabet member
 *     with a PWM row of its own) and any such symbol under the MotifSampler are
 *     GIBBS_ERR_UNSUPPORTED
 *   - base order of every 4-wide table: A, C, G, T
 *   - (float*int)[] results: parallel arrays double score[n] (log2, fs:303) and int32 site[n]
 *   - there is NO CPU fallback: every compute entry point launches CUDA kernels on the handle's
 *     device and fails with GIBBS_ERR_CUDA if that is impossible
 */
#ifndef GIBBS_B200_H
#define GIBBS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GIBBS_ABI_VERSION 2
#define GIBBS_MAX_K 32          /* motif width limit of the packed 64-bit window register      */
#define GIBBS_MAX_LEN (1 << 20) /* longest sequence                                            */

typedef enum gibbs_status {
    GIBBS_OK = 0,
    GIBBS_ERR_ARG = 1,         /* ArgumentNullException / ArgumentException (fs:24, fs:183)        */
    GIBBS_ERR_SYMBOL = 2,      /* IndexOutOfRangeException: symbol outside '*'..'Z' (fs:17, fs:20)   */
    GIBBS_ERR_SHORT_SEQ = 3,   /* InvalidOperationException from Array.take when L < k (fs:152)     */
    GIBBS_ERR_CUDA = 4,        /* CUDA runtime / launch failure or no usable device                 */
    GIBBS_ERR_NCCL = 5,        /* reserved: the one-process multi-device calls need no collective; one process */
                               /* per GPU uses the host layer's all_gather (torch.distributed)      */
    GIBBS_ERR_NOMEM = 6,       /* host or device allocation failed                                  */
    GIBBS_ERR_ROULETTE = 7,    /* ArgumentException of fs:753: pick beyond the accumulated mass     */
    GIBBS_ERR_UNSUPPORTED = 8  /* a mode outside the built hot path (see DESIGN.md, out of scope)   */
} gibbs_status;

/* sampler: which reference pipeline one chain (= one restart) runs */
#define GIBBS_SITE_SAMPLER 0  /* SiteSampler.doSiteSamplingWithBPV, fs:691-695                    */
#define GIBBS_MOTIF_SAMPLER 1 /* MotifSampler restart with fixed pcv, fs:876-879, motifAmount = 1 */

/* uniform source */
#define GIBBS_RNG_PHILOX 0    /* Philox4x32-10(key = seed, counter = (draw/4, chain)), u = word * 2^-32 */
#define GIBBS_RNG_INJECTED 1  /* caller-supplied doubles in [0,1): uniforms[chain][draw]                */

typedef struct gibbs_params {
    int32_t k;             /* motifLength                                                       */
    int32_t alphabet_size; /* alphabet.Length: the |A| of every pseudocount denominator (fs:257) */
    double pseudocount;    /* pseudoCount                                                       */
    double bg[4];          /* pcv.[A], pcv.[C], pcv.[G], pcv.[T] of the WithBPV family (fs:301)  */
    double cutoff;         /* MotifSampler cutOff (log2), fs:735                                */
    int32_t sampler;       /* GIBBS_SITE_SAMPLER | GIBBS_MOTIF_SAMPLER                          */
    int32_t phase_shifts;  /* SiteSampler: 1 = run the left/right shift sweeps (fs:694-695)     */
    int32_t max_sweeps;    /* safety cap per phase (the reference has none); 0 = 1000000        */
    int32_t phase_mask;    /* 0 = the whole pipeline of `sampler`; else a set of GIBBS_PHASE_* bits,  */
                           /* run in pipeline order from the state given to gibbs_set_start_state    */
    int32_t background;    /* GIBBS_BG_FIXED: bg[] (WithBPV family) | GIBBS_BG_DATA: derived from the */
                           /* sequences like doSiteSampling does (fs:697; per-window counts, fs:470)  */
    int32_t motif_amount;  /* MotifSampler motifAmount: sites per sequence, 0 / 1 = one, 2 = up to two (fs:727-742);  */
                           /* three and more are GIBBS_ERR_UNSUPPORTED                                */
} gibbs_params;

#define GIBBS_BG_FIXED 0
#define GIBBS_BG_DATA 1

/* phases = the reference functions a pipeline is made of */
#define GIBBS_PHASE_INIT 1        /* getPWMOfRandomStartsWithBPV, fs:412-430                          */
#define GIBBS_PHASE_GREEDY 2      /* findBestMotifWithStartPosition, fs:381-408                       */
#define GIBBS_PHASE_LEFT 4        /* getLeftShiftedBestPWMSsWithBPV, fs:350-377                       */
#define GIBBS_PHASE_RIGHT 8       /* getRightShiftedBestPWMSsWithBPV, fs:318-346                      */
#define GIBBS_PHASE_STOCHASTIC 16 /* findBestMotifPositionsWithStartPositionsByPCV, fs:828-853        */
#define GIBBS_PHASE_MOTIF_GREEDY 32 /* findBestMotifPositionsWithStartPositionByPCV, fs:788-822       */

typedef struct gibbs_run_stats {
    int64_t site_updates;  /* scans of one held-out sequence, all chains                        */
    int64_t window_scores; /* windows scored inside those scans                                 */
    int64_t sweeps;        /* passes n = 0..N-1, all chains                                     */
    int64_t exact_rescans; /* site updates that scored every window in float64 (no ranking pass) */
    int64_t capped_chains; /* chains stopped by max_sweeps                                      */
    int64_t speculative_discards; /* greedy-sweep site updates computed ahead and thrown away   */
    int32_t kernel_launches; /* CUDA kernels launched by the call                               */
    int32_t fast_path;     /* 1 = fixed-point filter + float64 verification was usable          */
    int32_t team_warps;    /* warps per chain of the first launch (1, 4, 8 or 16)               */
    int32_t init_path;     /* where the random starts ran: GIBBS_INIT_CHAIN / _WIDE / _SMEM / _TILED */
    double kernel_ms;      /* device time of the chain kernel (CUDA events on the handle stream) */
} gibbs_run_stats;

typedef struct gibbs_handle gibbs_handle;

/* ---- lifetime ------------------------------------------------------------------------------- */
int32_t gibbs_abi_version(void);
/* message of the most recent failure on this thread (never NULL) */
const char *gibbs_last_error(void);
/* number of CUDA devices visible, or 0 */
int32_t gibbs_device_count(void);

/*
 * Replaces: the `sources : BioArray<#IBioItem>[]` argument of every reference entry point
 * (fs:615, fs:691, fs:973 ...). Validates and uploads the sequences, 2-bit packs them on the GPU
 * (one row per sequence, rows padded to 16 B for bulk copies) and keeps them resident in HBM.
 */
int32_t gibbs_create(const uint8_t *seqs, const int64_t *offsets, int32_t n_seqs, int32_t device,
                     gibbs_handle **out);
/* replace the sequences of an existing handle (re-upload + re-pack, reusing device capacity) */
int32_t gibbs_upload(gibbs_handle *h, const uint8_t *seqs, const int64_t *offsets, int32_t n_seqs);
int32_t gibbs_destroy(gibbs_handle *h);
/* run all work of this handle on an existing CUDA stream (cudaStream_t as void*; NULL = own stream) */
int32_t gibbs_set_stream(gibbs_handle *h, void *cuda_stream);
int32_t gibbs_num_sequences(const gibbs_handle *h);
/* tuning knob: warps per chain, 1 / 4 / 8 / 16. 0 = automatic: 4 warps while many chains run, the last
 * 4 (1) chains per SM are handed over to launches with 8 (16) warps per chain */
int32_t gibbs_set_team_warps(gibbs_handle *h, int32_t warps);
int32_t gibbs_synchronize(gibbs_handle *h);
/*
 * Explicit per-handle switches for tests and measurements (no environment variable changes what a caller gets).
 * None of them changes a result.
 *   GIBBS_OPT_INIT_PATH    where the random starts (fs:412-430) run: GIBBS_INIT_AUTO (default) picks per launch;
 *                          _CHAIN = inside the chain kernel, _WIDE = grid-wide kernel gathering from global memory,
 *                          _SMEM = grid-wide kernel with the packed set in shared memory (used only when it fits),
 *                          _TILED = grid-wide kernel streaming the packed set through shared memory in tiles (large sets)
 *   GIBBS_OPT_EXACT_SCANS  1 = no ranking pass anywhere: every window in float64, sequential roulette walk
 *   GIBBS_OPT_STAGE2_AT / GIBBS_OPT_STAGE3_AT  straggler hand-over of the SiteSampler chain kernel: once this many chains
 *                          per SM (or fewer) are still running they continue with 8 / 16 warps per chain (defaults 4, 1)
 *   GIBBS_OPT_MIN_WIDTH    narrowest speculative round of the greedy sweeps while chains share an SM (default: the team size when
 *                          the first sweep runs on its own one-warp stage, else 1; once a
 *                          chain has an SM or a cluster to itself its rounds always use the whole team)
 *   GIBBS_OPT_CLUSTER      largest thread-block cluster the last stages may give one chain: 8 (default), 4 or 0 (none)
 *   GIBBS_OPT_SEQ_SWEEPS   how many of a restart's first sweeps run with one warp per chain before the team stages take over
 *                          (default 1: the first greedy sweep is sequential, a lone warp with more registers runs it faster
 *                          than a team that mostly waits; 0 = teams from the start; at most 3)
 *   GIBBS_OPT_TILE_ROWS    cap on the sequences per shared-memory tile of the _TILED random starts (0 = as many as fit)
 */
#define GIBBS_OPT_INIT_PATH 1
#define GIBBS_OPT_EXACT_SCANS 2
#define GIBBS_OPT_STAGE2_AT 3
#define GIBBS_OPT_STAGE3_AT 4
#define GIBBS_OPT_CLUSTER 5
#define GIBBS_OPT_MIN_WIDTH 6
#define GIBBS_OPT_TILE_ROWS 7
#define GIBBS_OPT_SEQ_SWEEPS 8
#define GIBBS_INIT_AUTO 0
#define GIBBS_INIT_CHAIN 1
#define GIBBS_INIT_WIDE 2
#define GIBBS_INIT_SMEM 3
#define GIBBS_INIT_TILED 4
int32_t gibbs_set_option(gibbs_handle *h, int32_t option, int32_t value);

/* ---- primitives: parity can be checked at the level the reference composes them -------------- */
/*
 * Replaces: getSegment -> createPFMOf -> fusePositionFrequencyMatrices for the N-1 other
 * sequences (fs:149, fs:211, fs:218; call sites fs:392-396). sites[i] < 0 means "no site"
 * (MotifSampler Positions = []). counts_out is int32 [k][4]. Bit-exact.
 */
int32_t gibbs_loo_counts(gibbs_handle *h, const int32_t *sites, int32_t heldout, int32_t k,
                         int32_t *counts_out);
/*
 * Replaces: createPPMOf -> normalizePPM -> createPositionWeightMatrix -> calculateSegmentScoreBy
 * for every window of sources.[heldout] (fs:249-293, loop of fs:301-314). raw_out (nullable) gets
 * the float64 products, log2_out (nullable) their log2; both have L - k + 1 entries.
 */
int32_t gibbs_window_scores(gibbs_handle *h, const int32_t *sites, int32_t heldout,
                            const gibbs_params *p, double *raw_out, double *log2_out);
/* Replaces: getBestPWMSsWithBPV (fs:301-314): first strict maximum; returns (log2 max, argmax). */
int32_t gibbs_pick_argmax(gibbs_handle *h, const int32_t *sites, int32_t heldout,
                          const gibbs_params *p, double *score_out, int32_t *site_out);
/*
 * Replaces: calculateNormalizedSegmentScores (motifAmount = 1) |> rouletteWheelSelection u
 * (fs:759-784, fs:746-754). site_out = -1 when a background ("no site") entry is selected;
 * pwms_out = the PWMS of the selected MotifIndex.
 */
int32_t gibbs_pick_roulette(gibbs_handle *h, const int32_t *sites, int32_t heldout,
                            const gibbs_params *p, double u, double *pwms_out, int32_t *site_out);

/* ---- chains / restarts ------------------------------------------------------------------------ */
/*
 * Replaces: the `positionProbabilityMatrix` argument of getMotifsWithBestPWMSOfPPM (fs:644-661) and of its callers
 * doSiteSamplingWithPPM (fs:703), getBestInformationContentOfPPM (fs:664), doMotifSamplingWithPPM (fs:1028),
 * getBestPWMSsOfPPM (fs:1002). ppm = double [k][4]: rows A,C,G,T of the reference's 49 x k matrix, entry j*4+b.
 * While set, the random starts (GIBBS_PHASE_INIT) of runs with GIBBS_BG_DATA and params.k == k are scored against
 * this PPM instead of the PPM of the random sites; the random sites still shape the background (fs:651-659) and
 * consume the same N(N-1) uniforms. ppm = NULL clears it. Runs with GIBBS_BG_FIXED reject a set PPM (the reference
 * has no such function).
 */
int32_t gibbs_set_start_ppm(gibbs_handle *h, const double *ppm_or_null, int32_t k);
/*
 * Start state for pipelines whose phase_mask lacks GIBBS_PHASE_INIT: the `startPositions :
 * (float*int)[]` / `motifMem : MotifIndex[]` argument of the sweep functions (fs:381, fs:350, fs:318,
 * fs:788, fs:828). sites int32 [n_chains][n_seqs] (-1 = Positions []), scores double
 * [n_chains][n_seqs]. Consumed by the next gibbs_run_device with the same n_chains.
 */
int32_t gibbs_set_start_state(gibbs_handle *h, int32_t n_chains, const int32_t *sites,
                              const double *scores);
/*
 * Replaces: one restart pipeline per chain --
 *   sampler 0, background 0: getPWMOfRandomStartsWithBPV |> findBestMotifWithStartPosition
 *              |> getLeftShiftedBestPWMSsWithBPV |> getRightShiftedBestPWMSsWithBPV (doSiteSamplingWithBPV, fs:691-695)
 *   sampler 0, background 1: the same pipeline over getBestPWMSs with the drifting background
 *              (doSiteSampling, fs:697-701; doSiteSamplingWithPPM, fs:703-707, after gibbs_set_start_ppm)
 *   sampler 1, background 0: getPWMOfRandomStartsWithBPV |> findBestMotifPositionsWithStartPositionsByPCV
 *              |> findBestMotifPositionsWithStartPositionByPCV, motifAmount = 1 (fs:876-879)
 *   sampler 1, background 1: doMotifSampling (fs:1034-1038) / doMotifSamplingWithPPM (fs:1028-1032), motifAmount = 1
 * n_chains independent chains (= restarts) run concurrently, a team of warps each; chain c uses the uniform stream
 * (seed, chain_id_base + c) or uniforms[c * uniforms_per_chain ...], so its result does not depend on how many
 * chains, launches or GPUs share the run. Draw order inside a chain: random init n ascending, i ascending skipping
 * n (fs:595-598), then one draw per n for the stochastic sweep (fs:851). Results stay on the device until gibbs_fetch.
 */
int32_t gibbs_run_device(gibbs_handle *h, const gibbs_params *p, int32_t n_chains,
                         int64_t chain_id_base, uint64_t seed, int32_t rng_mode,
                         const double *uniforms_or_null, int64_t uniforms_per_chain);
/*
 * Copies the results of the last gibbs_run_device to host buffers (any may be NULL):
 *   sites_out  int32 [n_chains][n_seqs]   (-1 = no site, MotifSampler only)
 *   scores_out double [n_chains][n_seqs]  log2 score / PWMS per sequence
 *   sums_out   double [n_chains]          Array.sum of the scores, left to right (fs:445)
 *   best_chain_out                        first chain with the largest sum (strict >, fs:450)
 *   counts_out int32 [k][4]               PWM counts (all N sites) of the best chain
 */
int32_t gibbs_fetch(gibbs_handle *h, int32_t *sites_out, double *scores_out, double *sums_out,
                    int32_t *best_chain_out, int32_t *counts_out, gibbs_run_stats *stats_out);
/*
 * Replaces: the promote-or-restart loop of getMotifsWithBestInformationContentWithBPV (fs:435-459; the same loop is
 * fs:616-640, fs:665-689, fs:857-881, fs:974-998; quirk A.6-8) over the restarts of the last gibbs_run_device, chain r
 * being restart r, with numberOfRepetitions = repetitions. The loop is decided on the device and only its result
 * crosses PCIe:
 *   sites_out  int32 [n_seqs], scores_out double [n_seqs]   the returned (float*int)[] / MotifIndex[]
 *   n_out      its length: n_seqs, or 1 when the loop's initial value [|(0., 0)|] survives
 *   sum_out    Array.sum of its scores; restart_out  which restart it is (-1 = the initial value)
 *   counts_out int32 [k][4]  PWM counts of its sites
 */
int32_t gibbs_fetch_best(gibbs_handle *h, int32_t repetitions, int32_t *sites_out, double *scores_out,
                         int32_t *n_out, double *sum_out, int32_t *restart_out, int32_t *counts_out,
                         gibbs_run_stats *stats_out);
/* gibbs_run_device + gibbs_fetch */
int32_t gibbs_run(gibbs_handle *h, const gibbs_params *p, int32_t n_chains, int64_t chain_id_base,
                  uint64_t seed, int32_t rng_mode, const double *uniforms_or_null,
                  int64_t uniforms_per_chain, int32_t *sites_out, double *scores_out,
                  double *sums_out, int32_t *best_chain_out, int32_t *counts_out,
                  gibbs_run_stats *stats_out);
/*
 * MotifIndex.Positions for motif_amount = m (fs:712-716): int32 [n_chains][n_seqs][m], newest position first -- the cons
 * order of fs:736, e.g. [306; 7] -- and -1 for an absent entry. sites_out of gibbs_fetch / gibbs_fetch_best holds the
 * first element of each list. gibbs_fetch_best_positions: the lists of the array the last gibbs_fetch_best returned,
 * int32 [n_seqs][m].
 */
int32_t gibbs_fetch_positions(gibbs_handle *h, int32_t m, int32_t *positions_out);
int32_t gibbs_fetch_best_positions(gibbs_handle *h, int32_t m, int32_t *positions_out);
/* gibbs_set_start_state for MotifIndex[] start states whose Positions hold up to m sites: positions int32
 * [n_chains][n_seqs][m] (newest first, -1 = absent), pwms double [n_chains][n_seqs] */
int32_t gibbs_set_start_motif_state(gibbs_handle *h, int32_t n_chains, int32_t m, const int32_t *positions,
                                    const double *pwms);
/* device pointers of the last run, for zero-copy collectives in the host layer (may be NULL) */
int32_t gibbs_device_results(gibbs_handle *h, void **sites_dev, void **scores_dev, void **sums_dev);

/* ---- one process, several devices ------------------------------------------------------------------------------ */
/*
 * Replaces: the restart axis the reference's author parallelised in the commented-out lines
 *   PSeq.map (fun _ -> doSiteSampling ...) (fsx:430)  /  PSeq.init 10 (fun _ -> doMotifSamplingWithPPM ...) (fsx:1162).
 * One handle per device with the sequences replicated on each; the restarts of a run are split into contiguous blocks
 * over the devices and run concurrently. Restart r uses the uniform stream (seed, chain_id_base + r) whatever device
 * it lands on, so results do not depend on the number of devices. No device-to-device traffic: the promote-or-restart
 * loop (fs:435-459) is decided on the host from one float64 sum per restart, then the winner's rows are fetched from
 * the device that holds them. (One process per GPU with a final NCCL all_gather is the other way to shard the same
 * axis; that is what bench.py --gpus N does through gibbssampling_b200/distributed.py.)
 * devices = NULL: devices 0 .. n_devices-1; n_devices = 0: every visible device.
 */
typedef struct gibbs_multi gibbs_multi;
int32_t gibbs_multi_create(const uint8_t *seqs, const int64_t *offsets, int32_t n_seqs, const int32_t *devices,
                           int32_t n_devices, gibbs_multi **out);
int32_t gibbs_multi_destroy(gibbs_multi *m);
int32_t gibbs_multi_num_devices(const gibbs_multi *m);
/* the handle of device slot i (for gibbs_set_option, gibbs_set_start_ppm ...); owned by m */
gibbs_handle *gibbs_multi_handle(gibbs_multi *m, int32_t i);
/* gibbs_run_device on every device: n_chains restarts in total */
int32_t gibbs_multi_run_device(gibbs_multi *m, const gibbs_params *p, int32_t n_chains, int64_t chain_id_base,
                               uint64_t seed, int32_t rng_mode, const double *uniforms_or_null,
                               int64_t uniforms_per_chain);
/* gibbs_fetch_best over the restarts of all devices (restart_out is the global restart index);
 * stats: counters summed over the devices, kernel_ms = the slowest device */
int32_t gibbs_multi_fetch_best(gibbs_multi *m, int32_t repetitions, int32_t *sites_out, double *scores_out,
                               int32_t *n_out, double *sum_out, int32_t *restart_out, int32_t *counts_out,
                               gibbs_run_stats *stats_out);

/* ---- many independent sequence sets in one launch ------------------------------------------------------------- */
/*
 * Replaces: a loop of getMotifsWithBestInformationContentWithBPV (fs:434-459) or getMotifsWithBestInformationContent
 * (fs:615-640) calls over many small sets, e.g. one discovery run per gene group or promoter region (fsx:223-365).
 * A batch holds S sets that share one gibbs_params; each set runs restarts_per_set restarts of the SiteSampler pipeline
 * and restart r of EVERY set uses the uniform stream (seed, chain_id_base + r). Set s gives bit for bit what a handle
 * created from set s alone gives for gibbs_run_device(h_s, p_s, restarts_per_set, chain_id_base, seed, GIBBS_RNG_PHILOX,
 * NULL, 0), p_s being p with bg = bg_per_set[s]. The restarts of all sets run in a few launches on one stream.
 * seqs / offsets as for gibbs_create over the concatenation of all sets; set s = sequences set_offsets[s] ..
 * set_offsets[s+1]-1 (int32 set_offsets[n_sets + 1], set_offsets[0] = 0, no empty set).
 * Errors follow the single-set rules per set and name the set (and sequence); a failed call leaves the batch usable.
 * The MotifSampler, phase_mask, start states, start PPMs and injected uniforms are not part of this API.
 */
typedef struct gibbs_batch gibbs_batch;
int32_t gibbs_batch_create(const uint8_t *seqs, const int64_t *offsets, const int32_t *set_offsets, int32_t n_sets,
                           int32_t device, gibbs_batch **out);
int32_t gibbs_batch_destroy(gibbs_batch *b);
/* restarts_per_set restarts of every set; bg_per_set double [n_sets][4] for GIBBS_BG_FIXED (NULL = p->bg for every set) */
int32_t gibbs_batch_run_device(gibbs_batch *b, const gibbs_params *p, const double *bg_per_set, int32_t restarts_per_set,
                               int64_t chain_id_base, uint64_t seed);
/* every restart of the last run (any may be NULL): sites_out int32 / scores_out double [sum_s R N_s], set-major then
 * restart-major (set s starts at R * set_offsets[s]); sums_out double [n_sets][R]; stats summed over the sets */
int32_t gibbs_batch_fetch(gibbs_batch *b, int32_t *sites_out, double *scores_out, double *sums_out, gibbs_run_stats *stats_out);
/* the promote-or-restart loop (fs:435-459) of every set, decided on the device (see gibbs_fetch_best); any may be NULL:
 * sites_out int32 / scores_out double [sum_s N_s] (set s at set_offsets[s], n_out[s] entries valid), n_out int32 [n_sets],
 * sum_out double [n_sets], restart_out int32 [n_sets] (-1 = the initial value), counts_out int32 [n_sets][k][4] */
int32_t gibbs_batch_fetch_best(gibbs_batch *b, int32_t repetitions, int32_t *sites_out, double *scores_out, int32_t *n_out,
                               double *sum_out, int32_t *restart_out, int32_t *counts_out, gibbs_run_stats *stats_out);

/* ---- host buffers ------------------------------------------------------------------------------- */
/* Page-locked host memory for the *_out arrays above (results of 1024 chains x 1000 sequences are
 * 12 MB; into pageable memory the copy is staged by the driver and pays first-touch page faults).
 * The reference keeps its results in GC arrays (fs:408 Array.copy); the shim may instead hand out
 * spans over these buffers. Any host pointer is accepted by every call; this is only faster. */
int32_t gibbs_host_alloc(size_t bytes, void **ptr_out);
int32_t gibbs_host_free(void *ptr);

/* ---- measurement support ------------------------------------------------------------------------ */
/* Streams `bytes` of shared-memory loads per SM for `iters` rounds; returns the achieved GB/s. */
int32_t gibbs_measure_smem_bandwidth(int32_t device, int32_t iters, double *gbps_out,
                                     double *ms_out);

#ifdef __cplusplus
}
#endif
#endif /* GIBBS_B200_H */
