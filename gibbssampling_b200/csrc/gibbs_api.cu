// gibbssampling_b200/csrc/gibbs_api.cu -- extern "C" boundary of libgibbs_b200.so (include/gibbs_b200.h).
//
// Host side of the drop-in: owns device memory and a stream, validates arguments the way the
// reference's exceptions would fire (SURVEY.md section 8b), launches the sm_100a kernels. There is no
// CPU implementation of any compute path in this file: without a CUDA device every compute entry
// point returns GIBBS_ERR_CUDA.
#include "../../include/gibbs_b200.h"
#include "gibbs_kernels.cuh"
#include "gibbs_motif.cuh"
#include "gibbs_motif2.cuh"
#include "gibbs_drift.cuh"
#include "gibbs_batch.cuh"
#include "gibbs_motif_batch.cuh"
#include "gibbs_fetch.cuh"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <type_traits>
#include <vector>

namespace gibbs { // gibbs_chain_tu.cu, one translation unit per group of chain_kernel instantiations (_build.py)
#define GIBBS_CHAIN_TU(name) cudaError_t name(const ChainArgs &a, int grid, int smem, cudaStream_t stream)
GIBBS_CHAIN_TU(launch_chain_t1);
GIBBS_CHAIN_TU(launch_chain_t4);
GIBBS_CHAIN_TU(launch_chain_t8);
GIBBS_CHAIN_TU(launch_chain_t16);
GIBBS_CHAIN_TU(launch_chain_masked_t1);
GIBBS_CHAIN_TU(launch_chain_masked_t4);
GIBBS_CHAIN_TU(launch_chain_masked_drift_t1);
GIBBS_CHAIN_TU(launch_chain_masked_drift_t4);
GIBBS_CHAIN_TU(launch_chain_drift_t1);
GIBBS_CHAIN_TU(launch_chain_drift_t4);
GIBBS_CHAIN_TU(launch_chain_drift_t8);
GIBBS_CHAIN_TU(launch_chain_init_t4);   // chain_kernel<.., INIT_ONLY>: the random starts on the chain's own team
GIBBS_CHAIN_TU(launch_chain_init_t1);
GIBBS_CHAIN_TU(launch_chain_init_drift_t4);
GIBBS_CHAIN_TU(launch_chain_init_drift_t1);
GIBBS_CHAIN_TU(launch_chain_init_masked_t4);
GIBBS_CHAIN_TU(launch_chain_init_masked_t1);
GIBBS_CHAIN_TU(launch_chain_init_masked_drift_t4);
GIBBS_CHAIN_TU(launch_chain_init_masked_drift_t1);
GIBBS_CHAIN_TU(launch_init_wide);       // gibbs_init_tu.cu: the grid-wide random-start kernels
GIBBS_CHAIN_TU(launch_init_wide_drift);
GIBBS_CHAIN_TU(launch_init_smem);
#undef GIBBS_CHAIN_TU
cudaError_t launch_init_tiled(const ChainArgs &a, int grid, int smem, cudaStream_t stream, int tile_rows); // gibbs_init_tu.cu
cudaError_t launch_motif_t4(const MotifArgs &m, int grid, int smem, cudaStream_t stream); // gibbs_motif_tu.cu
cudaError_t launch_motif_t1(const MotifArgs &m, int grid, int smem, cudaStream_t stream);
cudaError_t launch_motif_t8(const MotifArgs &m, int grid, int smem, cudaStream_t stream);  // hand-over stages
cudaError_t launch_motif_t16(const MotifArgs &m, int grid, int smem, cudaStream_t stream);
cudaError_t launch_motif_masked_t4(const MotifArgs &m, int grid, int smem, cudaStream_t stream); // symbols outside A,C,G,T
cudaError_t launch_motif_masked_t1(const MotifArgs &m, int grid, int smem, cudaStream_t stream);
cudaError_t launch_motif2(const Motif2Args &q, int grid, int smem, cudaStream_t stream); // gibbs_motif2_tu.cu
cudaError_t launch_motif2_seed(const int32_t *sites, long long cells, int32_t *pos2, cudaStream_t stream);
// gibbs_cluster_tu.cu: one chain on a cluster of 4 / 8 CTAs (capacity_out != null: only report how many clusters fit)
cudaError_t launch_chain_cluster4(const ChainArgs &a, int n_clusters, cudaStream_t stream, int *capacity_out);
cudaError_t launch_chain_cluster8(const ChainArgs &a, int n_clusters, cudaStream_t stream, int *capacity_out);
size_t launch_chain_cluster4_smem(int n, int row_words);
size_t launch_chain_cluster8_smem(int n, int row_words);
// gibbs_batch_tu.cu: chain_batch_kernel, one unit per (random starts only, masked symbols, drifting background, warps per chain)
#define GIBBS_BATCH_TU(name) cudaError_t name(const ChainArgs &run, const BatchTable &bt, int grid, int smem, cudaStream_t stream)
GIBBS_BATCH_TU(launch_batch_t4); GIBBS_BATCH_TU(launch_batch_t1);
GIBBS_BATCH_TU(launch_batch_drift_t4); GIBBS_BATCH_TU(launch_batch_drift_t1);
GIBBS_BATCH_TU(launch_batch_masked_t4); GIBBS_BATCH_TU(launch_batch_masked_t1);
GIBBS_BATCH_TU(launch_batch_masked_drift_t4); GIBBS_BATCH_TU(launch_batch_masked_drift_t1);
GIBBS_BATCH_TU(launch_batch_init_t4); GIBBS_BATCH_TU(launch_batch_init_t1);
GIBBS_BATCH_TU(launch_batch_init_drift_t4); GIBBS_BATCH_TU(launch_batch_init_drift_t1);
GIBBS_BATCH_TU(launch_batch_init_masked_t4); GIBBS_BATCH_TU(launch_batch_init_masked_t1);
GIBBS_BATCH_TU(launch_batch_init_masked_drift_t4); GIBBS_BATCH_TU(launch_batch_init_masked_drift_t1);
#undef GIBBS_BATCH_TU
// gibbs_motif_batch_tu.cu: motif_batch_kernel, one unit per (masked symbols, warps per restart); motif2_batch_kernel
#define GIBBS_MOTIF_BATCH_TU(name) cudaError_t name(const MotifArgs &run, const MotifBatchTable &bt, int grid, int smem, cudaStream_t stream)
GIBBS_MOTIF_BATCH_TU(launch_motif_batch_t4); GIBBS_MOTIF_BATCH_TU(launch_motif_batch_t1);
GIBBS_MOTIF_BATCH_TU(launch_motif_batch_masked_t4); GIBBS_MOTIF_BATCH_TU(launch_motif_batch_masked_t1);
GIBBS_MOTIF_BATCH_TU(launch_motif2_batch);
#undef GIBBS_MOTIF_BATCH_TU
}

using namespace gibbs;

namespace {

thread_local char g_err[512] = "";

int32_t fail(int32_t code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                                     \
    do {                                                                                                   \
        cudaError_t e_ = (expr);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return fail(e_ == cudaErrorMemoryAllocation ? GIBBS_ERR_NOMEM : GIBBS_ERR_CUDA, "%s: %s", #expr, \
                        cudaGetErrorString(e_));                                                           \
    } while (0)

// Device buffer owned by a handle. The owner's destroy function makes the handle's device current before the
// destructors run.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0; // elements
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
};

} // namespace

struct gibbs_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;

    int32_t n = 0, row_words = 0, max_len = 0, min_len = 0;
    DevBuf<uint8_t> ascii;
    DevBuf<int64_t> off;
    DevBuf<uint32_t> packed;
    DevBuf<uint32_t> mask;     // same geometry as packed: 0b01 at Gap '-', 0b11 at the other symbols outside A,C,G,T
    DevBuf<int32_t> rowflag;   // [n] sequence holds such a symbol
    DevBuf<uint64_t> wide;     // gather copy of the packed rows (DeviceSeqs::wide), built on first use
    bool wide_valid = false;
    int32_t wide_words = 0;
    DevBuf<int32_t> len;
    DevBuf<int> flags;    // [1..3] wtab range
    DevBuf<int> symflags; // pack_kernel: [0] 1 + byte outside '*'..'Z', [1] symbols outside A,C,G,T, [2] Gaps among them
    int64_t n_masked = 0;      // symbols outside A,C,G,T in the uploaded set
    bool has_gap = false;
    int64_t n_gap = 0;         // Gaps '-' among them (the Gap slot of the set totals when Gap is in the alphabet)

    // PWM value table, keyed by the parameters it was built for
    DevBuf<WEnt> wtab;
    bool wtab_valid = false;
    double wt_pc = 0, wt_bg[4] = {0, 0, 0, 0};
    int32_t wt_alen = 0;
    int wt_min = 0, wt_max = 0, wt_abnormal = 0;

    // primitive scratch
    DevBuf<int32_t> prim_sites;
    DevBuf<int32_t> prim_i32;
    DevBuf<double> prim_f64;

    // chain results
    DevBuf<int32_t> sites;
    DevBuf<double> hv, scores, sums;
    DevBuf<double> uniforms;
    DevBuf<unsigned long long> stats;
    DevBuf<int32_t> best; // [0] best chain, [1..] counts k*4
    int32_t run_chains = 0, run_k = 0, run_fast = 0, run_launches = 0;
    bool run_done = false;
    int32_t start_chains = 0; // chains covered by gibbs_set_start_state (0 = none pending)
    // MotifSampler: background-only window probabilities (depend on sequences, k and pcv only)
    DevBuf<double> bg_g, bg_sum, bg_max, cand_l;
    DevBuf<int32_t> bg_max_i, cand_w, err_flag;
    bool bg_valid = false;
    int32_t bg_k = 0, bg_wstride = 0;
    double bg_q[4] = {0, 0, 0, 0};
    int32_t run_sampler = 0;
    // data-derived background (doSiteSampling): normalizePPM values per count, base counts per sequence
    DevBuf<double> pvals, gbuf;
    DevBuf<double> start_ppm;  // gibbs_set_start_ppm: [k][4]
    int32_t start_ppm_k = 0;   // 0 = none set
    DevBuf<int32_t> basecnt, maskcnt;
    DevBuf<int32_t> ss;        // prefix tables [n][max_len + 2][4] of the ranking pass (null-sized when too large)
    bool ss_valid = false;
    bool drift_valid = false;
    double drift_pc = 0;
    int32_t drift_alen = 0;
    int32_t gcnt[4] = {0, 0, 0, 0};
    DevBuf<int32_t> ctl, resume, pending; // pause / resume of straggler chains
    int32_t run_extra_launches = 0;
    int32_t team_warps = 0;   // 0 = choose per launch; 1, 4, 8 or 16 = forced (gibbs_set_team_warps)
    int32_t run_team = 0;
    int sm_count = 0;
    std::vector<int32_t> len_host;     // sequence lengths (known from the offsets at upload: no read-back needed)
    int32_t start_max_excess = 0;      // max over the staged start sites of (site - length of its sequence)
    int32_t opt_init_path = 0;         // gibbs_set_option(GIBBS_OPT_INIT_PATH)
    int32_t opt_exact_scans = 0;       // gibbs_set_option(GIBBS_OPT_EXACT_SCANS)
    int32_t opt_stage2_at = 4, opt_stage3_at = 1; // hand-over thresholds in chains per SM (GIBBS_OPT_STAGE2_AT / _STAGE3_AT)
    int32_t opt_min_width = -1;        // GIBBS_OPT_MIN_WIDTH: -1 = automatic
    int32_t opt_seq_sweeps = 1;        // GIBBS_OPT_SEQ_SWEEPS: greedy sweeps run by one warp per chain before the team stages
    int32_t opt_tile_rows = 0;         // GIBBS_OPT_TILE_ROWS: cap on the sequences per tile of init_tiled_kernel (0 = what fits)
    int32_t opt_cluster = 8;           // largest cluster the last hand-over stages may use: 0 (none), 4 or 8 (GIBBS_OPT_CLUSTER)
    int32_t cluster_cap[2] = {-1, -1}; // clusters of 4 / 8 CTAs the device holds at once (queried once per shape)
    int32_t cluster_cap_n = 0, cluster_cap_rw = 0, cluster_cap_k = 0;
    int32_t wt_span = 0, drift_span = 0; // counts the W / PPM value tables cover: n (one site per sequence) or 2 n
    DevBuf<int32_t> pos2;              // motifAmount = 2: Positions [chains][n][2], newest first
    DevBuf<double> sc2;                // motifAmount = 2: window products of the current held-out sequence, per chain
    int32_t run_m = 1;                 // motifAmount of the last run
    int32_t start_m = 0;               // gibbs_set_start_motif_state staged Positions lists for this many sites (0 = none)
    bool best_valid = false;           // win_sites holds the winners of a fetch_best on the last run
    int32_t run_init_path = 0;         // where the random starts of the last run ran (GIBBS_INIT_*)
    DevBuf<int32_t> win_sites;         // fetch_winners: the winners' sites + [S] restart indices (+ [2 n] pair elements)
    DevBuf<double> win_scores;         // [n] winners' scores + [S] sums
    DevBuf<int32_t> counts;            // fetch_winners: PWM counts [m][S][k][4] of the winners' sites
    size_t smem_optin = 0;             // largest dynamic shared memory a block may opt in to
};

namespace {

int32_t set_device(const gibbs_handle *h) {
    CUDA_TRY(cudaSetDevice(h->device));
    return GIBBS_OK;
}

// Gap as an alphabet member has its PWM row for the SiteSampler with the data-derived background, where its background
// probability comes from the counts like a base's. The fixed background would need pcv.[Gap], which gibbs_params (bg[4])
// does not carry, and the MotifSampler has no Gap row in its tables.
bool gap_row_built(const gibbs_params *p) { return p->sampler == GIBBS_SITE_SAMPLER && p->background == GIBBS_BG_DATA; }

int32_t check_params(const gibbs_handle *h, const gibbs_params *p) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    if (!p) return fail(GIBBS_ERR_ARG, "null params");
    if (h->n < 1) return fail(GIBBS_ERR_ARG, "handle holds no sequences");
    if (p->k < 1 || p->k > GIBBS_MAX_K) return fail(GIBBS_ERR_ARG, "motif width k=%d outside 1..%d", p->k, GIBBS_MAX_K);
    if (h->min_len < p->k)
        return fail(GIBBS_ERR_SHORT_SEQ, "a sequence of length %d is shorter than k=%d (Array.take, fs:152)", h->min_len, p->k);
    if (p->alphabet_size < 1) return fail(GIBBS_ERR_ARG, "alphabet_size must be >= 1");
    if (!(p->pseudocount >= 0.0)) return fail(GIBBS_ERR_ARG, "pseudocount must be >= 0");
    if (p->background != GIBBS_BG_FIXED && p->background != GIBBS_BG_DATA) return fail(GIBBS_ERR_ARG, "unknown background mode %d", p->background);
    // An alphabet of >= 5 symbols is taken to hold Gap like the script's dnaBases (fsx:368-369). Gap then has
    // a PWM row of its own (quirk A.6-2); any other symbol outside A,C,G,T is not in the alphabet, has a PWM row
    // of 0 (fs:283-287) and is handled by the mask plane.
    if (h->has_gap && p->alphabet_size >= 5 && !gap_row_built(p))
        return fail(GIBBS_ERR_UNSUPPORTED, "sequences hold Gap '-' and alphabet_size = %d includes it: its PWM row is built for the "
                                           "SiteSampler with the data-derived background only (pass alphabet_size = 4 to score Gap "
                                           "like any other non-alphabet symbol)", p->alphabet_size);
    if (p->background == GIBBS_BG_FIXED)
        for (int b = 0; b < 4; ++b)
            if (!(p->bg[b] > 0.0)) return fail(GIBBS_ERR_ARG, "background probability bg[%d] must be > 0", b);
    return GIBBS_OK;
}

// normalizePPM of a set of n sequences: sum = float sourceCount + float alphabet.Length * pseudoCount (fs:257), with
// sourceCount = n - 1 sites
double ppm_den(int n, const gibbs_params *p) { return (double)(n - 1) + ((double)p->alphabet_size * p->pseudocount); }

// (re)build W(c, b) for c = 0..n-1 when the parameters it depends on changed
// span = how many counts the table covers: n, or 2 n when a sequence may contribute two sites (motifAmount = 2)
int32_t ensure_wtab(gibbs_handle *h, const gibbs_params *p, int *launches, int span_mult = 1) {
    const int span = h->n * span_mult;
    bool same = h->wtab_valid && h->wt_pc == p->pseudocount && h->wt_alen == p->alphabet_size && h->wt_span >= span;
    for (int b = 0; b < 4 && same; ++b) same = h->wt_bg[b] == p->bg[b];
    if (same) return GIBBS_OK;
    CUDA_TRY(h->wtab.reserve((size_t)span * 4));
    const int init[3] = {INT32_MAX, INT32_MIN, 0};
    CUDA_TRY(cudaMemcpyAsync(h->flags.p + 1, init, sizeof init, cudaMemcpyHostToDevice, h->stream));
    const double den = ppm_den(h->n, p);
    const int total = span * 4;
    wtab_kernel<<<(total + 255) / 256, 256, 0, h->stream>>>(span, p->pseudocount, den, p->bg[0], p->bg[1], p->bg[2],
                                                           p->bg[3], h->wtab.p, h->flags.p + 1);
    CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    int out[3];
    CUDA_TRY(cudaMemcpyAsync(out, h->flags.p + 1, sizeof out, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    h->wt_min = out[0];
    h->wt_max = out[1];
    h->wt_abnormal = out[2];
    h->wt_pc = p->pseudocount;
    h->wt_alen = p->alphabet_size;
    h->wt_span = span;
    memcpy(h->wt_bg, p->bg, sizeof h->wt_bg);
    h->wtab_valid = true;
    return GIBBS_OK;
}

// The fixed-point ranking pass is valid when no partial product of k table entries can leave the
// normal float64 range (and so the int32 key cannot overflow): |k * extreme log2| < 1000.
int fast_path_ok_range(int abnormal, int wt_min, int wt_max, int k) {
    if (abnormal) return 0;
    const double unit = 1.0 / (double)(1 << LG_FRAC_BITS);
    const double lo = (double)k * (wt_min < 0 ? wt_min : 0) * unit;
    const double hi = (double)k * (wt_max > 0 ? wt_max : 0) * unit;
    return (lo > -1000.0 && hi < 1000.0) ? 1 : 0;
}
int fast_path_ok(const gibbs_handle *h, int k) { return fast_path_ok_range(h->wt_abnormal, h->wt_min, h->wt_max, k); }

// The ranking pass of the drifting background is valid when every odds ratio ppm / pcv, which lies in [pc / den, den / pc]
// with den <= all bases of the set + one more sequence + |A| pc (or N - 1 + |A| pc), keeps every float64 product of k of
// them in the normal range (|log2| < 1000), and pc >= 1e-30 keeps every float32 logarithm argument normal and finite.
// gaps = the set's Gaps when Gap is in the alphabet (they enter every denominator), else 0.
int drift_fast_path_ok(const int32_t gcnt[4], int32_t gaps, int32_t max_len, int32_t n, const gibbs_params *p) {
    const double alpha_pc = (double)p->alphabet_size * p->pseudocount;
    const double bases = (double)gcnt[0] + gcnt[1] + gcnt[2] + gcnt[3] + (double)gaps + (double)max_len;
    const double den = (bases > (double)n ? bases : (double)n) + alpha_pc;
    return (p->pseudocount >= 1e-30 && (double)p->k * log2(den / p->pseudocount) < 1000.0) ? 1 : 0;
}

template <typename K>
int32_t set_smem(K kernel, int bytes) {
    if (bytes > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return GIBBS_OK;
}

#define KP_CASES(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16)

// f(std::integral_constant<int, KP>()) with KP = (k + 1) / 2, the template argument of the kernels that hold a k-mer
template <typename F>
int32_t with_kp(int k, F &&f) {
    switch ((k + 1) / 2) {
#define X(KPV) case KPV: return f(std::integral_constant<int, KPV>());
        KP_CASES(X)
#undef X
    default: return fail(GIBBS_ERR_ARG, "unsupported k");
    }
}

// one CTA of one warp with the staging buffers of a one-warp team (the primitives)
template <typename K, typename... A>
int32_t launch_one_warp(gibbs_handle *h, K kernel, int row_words, const A &...args) {
    const int smem = team_smem_bytes(row_words, 1);
    const int32_t rc = set_smem(kernel, smem);
    if (rc) return rc;
    kernel<<<1, 32, smem, h->stream>>>(args...);
    CUDA_TRY(cudaGetLastError());
    return GIBBS_OK;
}

// The unit of a kernel family (_build.py) that holds the instantiation for (warps per chain, masked symbols, drifting
// background, random starts only).
template <typename F>
struct Unit {
    int team, masked, drift, init;
    F launch;
};

template <typename F, size_t U>
int32_t find_unit(const Unit<F> (&units)[U], const char *family, int team, bool masked, bool drift, bool init, F *out) {
    for (const Unit<F> &u : units)
        if (u.team == team && u.masked == masked && u.drift == drift && u.init == init) {
            *out = u.launch;
            return GIBBS_OK;
        }
    return fail(GIBBS_ERR_ARG, "no %s kernel is built for %d warps per chain (masked symbols %d, drifting background %d, "
                               "random starts only %d)", family, team, masked, drift, init);
}

using ChainLaunch = cudaError_t (*)(const ChainArgs &, int, int, cudaStream_t);
const Unit<ChainLaunch> CHAIN_UNITS[] = {
    {1, 0, 0, 0, launch_chain_t1}, {4, 0, 0, 0, launch_chain_t4}, {8, 0, 0, 0, launch_chain_t8}, {16, 0, 0, 0, launch_chain_t16},
    {1, 0, 1, 0, launch_chain_drift_t1}, {4, 0, 1, 0, launch_chain_drift_t4}, {8, 0, 1, 0, launch_chain_drift_t8},
    {1, 1, 0, 0, launch_chain_masked_t1}, {4, 1, 0, 0, launch_chain_masked_t4},
    {1, 1, 1, 0, launch_chain_masked_drift_t1}, {4, 1, 1, 0, launch_chain_masked_drift_t4},
    {1, 0, 0, 1, launch_chain_init_t1}, {4, 0, 0, 1, launch_chain_init_t4},
    {1, 0, 1, 1, launch_chain_init_drift_t1}, {4, 0, 1, 1, launch_chain_init_drift_t4},
    {1, 1, 0, 1, launch_chain_init_masked_t1}, {4, 1, 0, 1, launch_chain_init_masked_t4},
    {1, 1, 1, 1, launch_chain_init_masked_drift_t1}, {4, 1, 1, 1, launch_chain_init_masked_drift_t4},
};

// the MotifSampler units serve both backgrounds and continue from the random starts wherever those ran
using MotifLaunch = cudaError_t (*)(const MotifArgs &, int, int, cudaStream_t);
const Unit<MotifLaunch> MOTIF_UNITS[] = {
    {1, 0, 0, 0, launch_motif_t1}, {4, 0, 0, 0, launch_motif_t4}, {8, 0, 0, 0, launch_motif_t8}, {16, 0, 0, 0, launch_motif_t16},
    {1, 1, 0, 0, launch_motif_masked_t1}, {4, 1, 0, 0, launch_motif_masked_t4},
};

using BatchLaunch = cudaError_t (*)(const ChainArgs &, const BatchTable &, int, int, cudaStream_t);
const Unit<BatchLaunch> BATCH_UNITS[] = {
    {1, 0, 0, 0, launch_batch_t1}, {4, 0, 0, 0, launch_batch_t4}, {1, 0, 1, 0, launch_batch_drift_t1}, {4, 0, 1, 0, launch_batch_drift_t4},
    {1, 1, 0, 0, launch_batch_masked_t1}, {4, 1, 0, 0, launch_batch_masked_t4},
    {1, 1, 1, 0, launch_batch_masked_drift_t1}, {4, 1, 1, 0, launch_batch_masked_drift_t4},
    {1, 0, 0, 1, launch_batch_init_t1}, {4, 0, 0, 1, launch_batch_init_t4},
    {1, 0, 1, 1, launch_batch_init_drift_t1}, {4, 0, 1, 1, launch_batch_init_drift_t4},
    {1, 1, 0, 1, launch_batch_init_masked_t1}, {4, 1, 0, 1, launch_batch_init_masked_t4},
    {1, 1, 1, 1, launch_batch_init_masked_drift_t1}, {4, 1, 1, 1, launch_batch_init_masked_drift_t4},
};

// motifAmount = 1; the units serve both backgrounds (motifAmount = 2: launch_motif2_batch)
using MotifBatchLaunch = cudaError_t (*)(const MotifArgs &, const MotifBatchTable &, int, int, cudaStream_t);
const Unit<MotifBatchLaunch> MOTIF_BATCH_UNITS[] = {
    {1, 0, 0, 0, launch_motif_batch_t1}, {4, 0, 0, 0, launch_motif_batch_t4},
    {1, 1, 0, 0, launch_motif_batch_masked_t1}, {4, 1, 0, 0, launch_motif_batch_masked_t4},
};

// one launch of the chain_kernel unit for (warps per chain, masked symbols, drifting background, random starts only)
int32_t launch_chain_unit(gibbs_handle *h, int team, bool masked, bool drift, bool init, const ChainArgs &a, int grid) {
    const int smem = team_smem_bytes(a.s.row_words, team);
    if (smem > 200 * 1024) return fail(GIBBS_ERR_ARG, "sequences too long for %d warps per chain", team);
    ChainLaunch f;
    const int32_t rc = find_unit(CHAIN_UNITS, "chain", team, masked, drift, init, &f);
    if (rc) return rc;
    CUDA_TRY(f(a, grid, smem, h->stream));
    return GIBBS_OK;
}

// Random starts are N independent site updates of N-1 draws each, so they need not run on the chain's own team:
//   GIBBS_INIT_SMEM   grid-wide, one CTA per SM holding the whole packed set in shared memory (the draws gather
//                     from LDS): whenever the set fits (fixed background, A,C,G,T only) -- C2: 144 KB
//   GIBBS_INIT_WIDE   grid-wide with global gathers: few chains or many sequences (C4, 8 chains: 17.2 s -> 0.61 s
//                     against the chain kernel's INIT sweep)
//   GIBBS_INIT_CHAIN  inside the chain kernel: many chains of few sequences whose set does not fit
// Launches the grid-wide kernel if one is chosen and clears GIBBS_PHASE_INIT from a.phase_mask.
int32_t launch_random_starts(gibbs_handle *h, ChainArgs &a, bool drift) {
    const bool masked = a.s.mask != nullptr; // symbols outside A,C,G,T: inside the MASKED chain kernel
    const int kp = (a.k + 1) / 2;
    int init_path = GIBBS_INIT_CHAIN, tile_rows = 0;
    if ((a.phase_mask & GIBBS_PHASE_INIT) && !masked) {
        const bool smem_ok = !drift && init_smem_total_bytes(a.s.n, a.s.row_words, kp) <= h->smem_optin;
        const bool smem_fits = smem_ok && (long long)a.n_chains * a.s.n >= (long long)h->sm_count * ISM_WARPS;
        const bool wide_fits = init_smem_bytes(a.s.row_words) <= 200 * 1024;
        const bool wide_wins = a.n_chains < 4 * h->sm_count || a.s.n >= 4096 || a.sampler == GIBBS_MOTIF_SAMPLER;
        init_path = smem_fits ? GIBBS_INIT_SMEM : (wide_fits && wide_wins) ? GIBBS_INIT_WIDE : GIBBS_INIT_CHAIN;
        // the set streamed through shared memory in tiles: the Philox stream, fixed background, at least 256 sequences per
        // tile; chosen by itself where the global gathers of the wide kernel are the limit (many sequences, work for every SM)
        tile_rows = (int)(((long long)h->smem_optin - 128 - 256 - (long long)TILED_WARPS * (ism_table_bytes(kp) + a.s.row_words * 4)) / 2
                          / ((long long)a.s.row_words * 4));
        const bool tile_auto = tile_rows >= 256;
        if (tile_rows > a.s.n) tile_rows = a.s.n;
        if (h->opt_tile_rows > 0 && tile_rows > h->opt_tile_rows) tile_rows = h->opt_tile_rows; // (tests: many small tiles)
        const bool tiled_ok = !drift && a.rng_mode == 0 && tile_rows >= 1; // (both samplers: the MotifSampler starts from the same sweep)
        if (init_path == GIBBS_INIT_WIDE && tiled_ok && tile_auto && a.s.n >= 4096 && (long long)a.n_chains * a.s.n >= 8LL * h->sm_count * TILED_WARPS)
            init_path = GIBBS_INIT_TILED;
        if (h->opt_init_path == GIBBS_INIT_CHAIN) init_path = GIBBS_INIT_CHAIN;
        if (h->opt_init_path == GIBBS_INIT_WIDE && wide_fits) init_path = GIBBS_INIT_WIDE;
        if (h->opt_init_path == GIBBS_INIT_SMEM && smem_ok) init_path = GIBBS_INIT_SMEM;
        if (h->opt_init_path == GIBBS_INIT_TILED && tiled_ok) init_path = GIBBS_INIT_TILED;
    }
    h->run_init_path = init_path;
    if (init_path == GIBBS_INIT_TILED) {
        const int smem = (int)init_tiled_total_bytes(tile_rows, a.s.row_words, kp);
        const long long items = (long long)a.n_chains * a.s.n;
        long long grid = (items + TILED_WARPS - 1) / TILED_WARPS;
        if (grid > h->sm_count) grid = h->sm_count;
        CUDA_TRY(launch_init_tiled(a, (int)grid, smem, h->stream, tile_rows));
        a.phase_mask &= ~GIBBS_PHASE_INIT; // the chain kernel continues from the state just written
        h->run_extra_launches += 1;
    } else
    if (init_path == GIBBS_INIT_SMEM) {
        const int smem = (int)init_smem_total_bytes(a.s.n, a.s.row_words, kp);
        const long long items = (long long)a.n_chains * a.s.n;
        long long grid = (items + ISM_WARPS - 1) / ISM_WARPS;
        if (grid > h->sm_count) grid = h->sm_count;
        CUDA_TRY(launch_init_smem(a, (int)grid, smem, h->stream));
        a.phase_mask &= ~GIBBS_PHASE_INIT; // the chain kernel continues from the state just written
        h->run_extra_launches += 1;
    } else if (init_path == GIBBS_INIT_WIDE) {
        if (!h->wide_valid && a.k <= 25 && !masked) { // the gather copy: 8 bytes per 8 bases, built once per upload
            const int ww = h->max_len / 8 + 1;
            const size_t words = (size_t)h->n * ww;
            if (words * 8 <= ((size_t)8 << 30) && h->wide.reserve(words) == cudaSuccess) {
                wide_kernel<<<(unsigned)((words + 255) / 256), 256, 0, h->stream>>>(h->packed.p, h->n, h->row_words, ww, h->wide.p);
                CUDA_TRY(cudaGetLastError());
                h->wide_words = ww;
                h->wide_valid = true;
                h->run_extra_launches += 1;
                a.s.wide = h->wide.p;
                a.s.wide_words = ww;
            } else {
                cudaGetLastError(); // not enough memory: the packed rows serve
            }
        }
        const int smem = init_smem_bytes(a.s.row_words);
        const long long items = (long long)a.n_chains * a.s.n;
        long long grid = (items + INIT_WARPS - 1) / INIT_WARPS;
        if (grid > 4LL * h->sm_count) grid = 4LL * h->sm_count;
        CUDA_TRY(drift ? launch_init_wide_drift(a, (int)grid, smem, h->stream) : launch_init_wide(a, (int)grid, smem, h->stream));
        a.phase_mask &= ~GIBBS_PHASE_INIT;
        h->run_extra_launches += 1;
    } else if (a.phase_mask & GIBBS_PHASE_INIT) { // on the chain's own team: one CTA of 4 warps (or 1) per chain
        const int team = (a.s.n >= 4 && team_smem_bytes(a.s.row_words, 4) <= 200 * 1024 && h->team_warps != 1) ? 4 : 1;
        ChainArgs b = a;
        b.from_list = 0;
        b.pause_below = 0;
        const int32_t rc = launch_chain_unit(h, team, masked, drift, true, b, a.n_chains);
        if (rc) return rc;
        a.phase_mask &= ~GIBBS_PHASE_INIT;
        h->run_extra_launches += 1;
    }
    return GIBBS_OK;
}

// One launch of a run. Its chains pause at their next sweep boundary once fewer than pause_below are still running
// (0 = run to the end) and the next stage continues them; cluster: CTAs per thread-block cluster (0 = one CTA per chain);
// min_sweeps: sweeps a chain runs in the stage before it may pause; min_width: ChainArgs::min_width.
struct Stage {
    int team, pause_below, cluster, min_sweeps, min_width;
};
constexpr int MAX_STAGES = 8; // the control words hold one count per stage

// The stages of a run of either sampler (a: after the random starts).
// Warps per chain. Four warps work on four consecutive held-out sequences of the chain at once, which
// shortens every chain's critical path (measured faster than one warp per chain both when all chains
// are resident at once -- C2 -- and when they run in several waves); one warp is kept for sets with
// fewer than 4 sequences or rows too long for four sets of staging buffers.
// Chains need very different numbers of sweeps, so a one-wave launch ends with a few chains running on a mostly idle GPU.
// Stage 1 runs every chain with 4 warps (7 chains per SM); once <= opt_stage2_at chains per SM are still running they
// pause at their next sweep boundary and stage 2 continues them with 8 warps; once <= opt_stage3_at chains per SM are
// left, stage 3 continues with 16 warps. Runs with fewer chains start on the wider teams: those are used only while warp
// slots are idle. Late sweeps move few sites, so the wider speculative rounds are rarely discarded.
int plan_stages(gibbs_handle *h, const ChainArgs &a, bool drift, Stage *stages) {
    const int N = a.s.n, sms = h->sm_count, chains = a.n_chains;
    const bool masked = a.s.mask != nullptr;
    auto fits = [&](int t) { return N >= t && team_smem_bytes(a.s.row_words, t) <= 200 * 1024; };
    auto widest_fit = [&](int t) { // 16 -> 8 -> 4 -> 1 warps
        while (t > 1 && !fits(t)) t = t > 4 ? t / 2 : 1;
        return t;
    };
    int n = 0;
    auto widen = [&](int at8, int at16) { // the last chains continue on 8, then on 16 warps (at16 = 0: no 16-warp stage)
        if (stages[n - 1].team == 4 && fits(8)) {
            stages[n - 1].pause_below = at8;
            stages[n++] = {8};
        }
        if (at16 > 0 && stages[n - 1].team == 8 && fits(16)) {
            stages[n - 1].pause_below = at16;
            stages[n++] = {16};
        }
    };
    const int at8 = h->opt_stage2_at * sms, at16 = h->opt_stage3_at * sms;
    const int first = widest_fit(chains > at8 ? 4 : chains > at16 ? 8 : 16);
    if (a.sampler == GIBBS_MOTIF_SAMPLER) {
        // (One warp per restart for the first greedy sweeps, as the SiteSampler runs them, was measured here too: the sweeps
        // themselves gain 1.4 ms on C2, the two hand-overs around them cost 2.5 ms -- tools/experiments/README.md.)
        if (masked || h->team_warps != 0 || !fits(4)) { // one stage (a forced team of 8 or 16 warps runs on 4)
            stages[n++] = {h->team_warps != 1 && fits(4) ? 4 : 1};
        } else {
            stages[n++] = {first};
            widen(at8, at16);
        }
        return n; // (min_width stays 0)
    }
    if (masked) { // one launch of the MASKED instantiation (1 or 4 warps)
        stages[n++] = {team_smem_bytes(a.s.row_words, 4) <= 200 * 1024 ? 4 : 1};
    } else if (drift) { // data-derived background: 4 warps per chain (4 chains per SM), the last 2 per SM continue with 8
        const int forced = h->team_warps == 16 ? 8 : h->team_warps;
        stages[n++] = {forced != 0 ? forced : widest_fit(chains > 2 * sms ? 4 : 8)};
        if (forced == 0) widen(2 * sms, 0);
    } else if (h->team_warps != 0) {
        stages[n++] = {h->team_warps};
    } else {
        // The first greedy sweep moves a site in almost every update (C2: 99 %, then 28 % in sweep 1), so its rounds run at
        // width 1 and three warps of a four-warp team wait. One warp per chain with 128 registers and no team barrier runs
        // such a sweep faster (C2, sweeps 0 / 1 / 2 / 3 alone: 1.74 / 1.61 / 1.57 / 1.52 ms against 2.20 / 2.18 / 1.59 / 1.15 ms,
        // tools/seq_regime_probe.py). So the first GIBBS_OPT_SEQ_SWEEPS sweeps are a stage of their own on
        // chain_kernel<KP, 1>: every chain pauses at the boundary of that sweep (pause_below = all chains) and the next
        // stage continues it. The hand-over itself costs ~0.3 ms (the slowest chain's sweep ends the launch), so whole C2
        // steps measure 23.76 / 23.18 / 23.48 / 24.2 ms for 0 / 1 / 2 / 3 such sweeps: the default is 1.
        if (first == 4 && N >= 64 && (a.phase_mask & GIBBS_PHASE_GREEDY) && h->opt_seq_sweeps > 0)
            stages[n++] = {1, chains, 0, h->opt_seq_sweeps};
        stages[n++] = {first};
        widen(at8, at16);
        // With fewer chains than SMs left, one chain gets several SMs: a thread-block cluster of 4, then 8 CTAs of 16 warps
        // (chain_cluster_kernel). Needs the ranking pass, the W table in shared memory and rounds of 64 sequences to fill.
        if (stages[n - 1].team == 16 && h->opt_cluster >= 4 && a.fast_ok && N >= 128) {
            if (h->cluster_cap_n != N || h->cluster_cap_rw != a.s.row_words || h->cluster_cap_k != a.k) {
                h->cluster_cap[0] = h->cluster_cap[1] = 0;
                int cap = 0;
                if (launch_chain_cluster4_smem(N, a.s.row_words) <= h->smem_optin &&
                    launch_chain_cluster4(a, 1, h->stream, &cap) == cudaSuccess) h->cluster_cap[0] = cap;
                cap = 0;
                if (launch_chain_cluster8_smem(N, a.s.row_words) <= h->smem_optin &&
                    launch_chain_cluster8(a, 1, h->stream, &cap) == cudaSuccess) h->cluster_cap[1] = cap;
                cudaGetLastError();
                h->cluster_cap_n = N; h->cluster_cap_rw = a.s.row_words; h->cluster_cap_k = a.k;
            }
            if (h->cluster_cap[0] > 0) {
                stages[n - 1].pause_below = h->cluster_cap[0];
                stages[n++] = {16, 0, 4};
                if (h->opt_cluster >= 8 && h->cluster_cap[1] > 0 && h->cluster_cap[1] < h->cluster_cap[0]) {
                    stages[n - 1].pause_below = h->cluster_cap[1];
                    stages[n++] = {16, 0, 8};
                }
            }
        }
    }
    for (int st = 0; st < n; ++st) {
        // chains that reach this stage per SM (at most): with an SM or more per chain, never narrow a speculative round
        const int per_sm = ((st == 0 ? chains : stages[st - 1].pause_below) + sms - 1) / sms;
        // Stages that share SMs (GIBBS_OPT_MIN_WIDTH): while the first sweep -- a mover in almost every update -- ran on the
        // teams, narrowing after a discarded round saved the other chains' issue slots (width 1). With that sweep on
        // stage 0 the remaining sweeps discard far less than they gain from never narrowing: C2 23.2 -> 22.6 ms.
        const bool seq_stage = stages[0].team == 1 && stages[0].min_sweeps > 0;
        stages[st].min_width = stages[st].cluster ? stages[st].cluster * 16 : per_sm <= 1 ? stages[st].team
                               : h->opt_min_width >= 1 ? h->opt_min_width : seq_stage ? stages[st].team : 1;
    }
    return n;
}

// Runs the stages of a plan. Sets up the control words and the lists through which each stage hands its paused chains to
// the next; launch(stage, args, grid) launches one stage on a grid of the chains the previous stage paused at most.
template <typename Launch>
int32_t run_stages(gibbs_handle *h, ChainArgs a, const Stage *stages, int n_stages, Launch &&launch) {
    h->run_team = stages[0].min_sweeps > 0 ? stages[1].team : stages[0].team; // (the team of the main stage)
    // control words: [0] chains still running, [s] number of chains paused by stage s
    CUDA_TRY(h->ctl.reserve(MAX_STAGES));
    const int32_t ctl0[MAX_STAGES] = {a.n_chains, 0, 0, 0, 0, 0, 0, 0};
    CUDA_TRY(cudaMemcpyAsync(h->ctl.p, ctl0, sizeof ctl0, cudaMemcpyHostToDevice, h->stream));
    a.active = h->ctl.p;
    if (n_stages > 1) {
        CUDA_TRY(h->resume.reserve((size_t)a.n_chains));
        CUDA_TRY(h->pending.reserve((size_t)(n_stages - 1) * (size_t)a.n_chains));
        a.resume = h->resume.p;
    }
    for (int st = 0; st < n_stages; ++st) {
        ChainArgs b = a;
        b.pause_below = stages[st].pause_below;
        b.pause_min_sweeps = stages[st].min_sweeps;
        b.min_width = stages[st].min_width;
        b.from_list = st > 0;
        b.pending_in = st > 0 ? h->pending.p + (size_t)(st - 1) * a.n_chains : nullptr;
        b.pending_in_n = st > 0 ? h->ctl.p + st : nullptr;
        b.pending_out = st + 1 < n_stages ? h->pending.p + (size_t)st * a.n_chains : nullptr;
        b.pending_out_n = st + 1 < n_stages ? h->ctl.p + st + 1 : nullptr;
        const int32_t rc = launch(stages[st], b, st == 0 ? a.n_chains : stages[st - 1].pause_below);
        if (rc) return rc;
        if (st > 0) h->run_extra_launches += 1;
    }
    return GIBBS_OK;
}

int32_t launch_chain(gibbs_handle *h, ChainArgs a, bool drift) {
    h->run_extra_launches = 0;
    int32_t rc = launch_random_starts(h, a, drift);
    if (rc) return rc;
    Stage stages[MAX_STAGES] = {};
    const int n_stages = plan_stages(h, a, drift, stages);
    const bool masked = a.s.mask != nullptr;
    return run_stages(h, a, stages, n_stages, [&](const Stage &s, const ChainArgs &b, int grid) -> int32_t {
        if (s.cluster == 0) return launch_chain_unit(h, s.team, masked, drift, false, b, grid);
        CUDA_TRY((s.cluster == 4 ? launch_chain_cluster4 : launch_chain_cluster8)(b, grid, h->stream, nullptr));
        return GIBBS_OK;
    });
}

// the stages of a MotifSampler run (m: after the random starts)
int32_t launch_motif(gibbs_handle *h, const MotifArgs &m, const Stage *stages, int n_stages) {
    const bool masked = m.c.s.mask != nullptr;
    return run_stages(h, m.c, stages, n_stages, [&](const Stage &s, const ChainArgs &c, int grid) -> int32_t {
        MotifLaunch f;
        const int32_t rc = find_unit(MOTIF_UNITS, "MotifSampler", s.team, masked, false, false, &f);
        if (rc) return rc;
        MotifArgs b = m;
        b.c = c;
        CUDA_TRY(f(b, grid, team_smem_bytes(c.s.row_words, s.team), h->stream));
        return GIBBS_OK;
    });
}

int32_t launch_loo_counts(gibbs_handle *h, const PrimArgs &a) {
    return with_kp(a.k, [&](auto kp) { return launch_one_warp(h, loo_counts_kernel<kp()>, a.s.row_words, a); });
}

int32_t launch_scan(gibbs_handle *h, const PrimArgs &a, int mode) {
    return with_kp(a.k, [&](auto kp) { return launch_one_warp(h, scan_kernel<kp()>, a.s.row_words, a, mode); });
}

int32_t launch_all_counts(gibbs_handle *h, const DeviceSeqs &s, const int32_t *sites, int k, int32_t *out) {
    return with_kp(k, [&](auto kp) { return launch_one_warp(h, all_counts_kernel<kp()>, s.row_words, s, sites, k, out); });
}

int32_t launch_roulette(gibbs_handle *h, const RouletteArgs &r) {
    return with_kp(r.p.k, [&](auto kp) { return launch_one_warp(h, roulette_kernel<kp()>, r.p.s.row_words, r); });
}

DeviceSeqs dev_seqs(const gibbs_handle *h);

int32_t ensure_bgtab(gibbs_handle *h, const gibbs_params *p, int *launches) {
    bool same = h->bg_valid && h->bg_k == p->k;
    for (int b = 0; b < 4 && same; ++b) same = h->bg_q[b] == p->bg[b];
    if (same) return GIBBS_OK;
    const int wstride = h->max_len - p->k + 1;
    CUDA_TRY(h->bg_g.reserve((size_t)h->n * wstride));
    CUDA_TRY(h->bg_sum.reserve((size_t)h->n));
    CUDA_TRY(h->bg_max.reserve((size_t)h->n));
    CUDA_TRY(h->bg_max_i.reserve((size_t)h->n));
    bg_setup_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(dev_seqs(h), p->k, p->bg[0], p->bg[1], p->bg[2], p->bg[3],
                                                                wstride, h->bg_g.p, h->bg_sum.p, h->bg_max.p, h->bg_max_i.p);
    CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    h->bg_k = p->k;
    h->bg_wstride = wstride;
    memcpy(h->bg_q, p->bg, sizeof h->bg_q);
    h->bg_valid = true;
    return GIBBS_OK;
}

// per sequence (any background parameters): A,C,G,T counts, symbols outside A,C,G,T, prefix tables of the ranking pass
int32_t ensure_seq_counts(gibbs_handle *h, int *launches) {
    CUDA_TRY(h->basecnt.reserve((size_t)h->n * 4));
    CUDA_TRY(h->maskcnt.reserve((size_t)h->n));
    basecount_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(dev_seqs(h), h->basecnt.p, h->maskcnt.p);
    CUDA_TRY(cudaGetLastError());
    // prefix tables of the ranking pass: int32 sums reach L^2 / 2, and 16 B per base are only worth keeping while they
    // fit comfortably (C4: 320 MB); otherwise the ranking pass keeps its sliding counters
    h->ss_valid = false;
    const size_t ss_ints = (size_t)h->n * (size_t)(h->max_len + 2) * 4;
    if (h->max_len <= 46000 && ss_ints * sizeof(int32_t) <= ((size_t)4 << 30)) {
        if (h->ss.reserve(ss_ints) == cudaSuccess) {
            prefix_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(dev_seqs(h), h->max_len + 2, reinterpret_cast<int4 *>(h->ss.p));
            if (launches) *launches += 1;
            h->ss_valid = true;
        } else {
            cudaGetLastError(); // not enough memory: fall back to the sliding counters
        }
    }
    CUDA_TRY(cudaGetLastError());
    if (launches) *launches += 1;
    return GIBBS_OK;
}

int32_t ensure_drift(gibbs_handle *h, const gibbs_params *p, int *launches, int span_mult = 1) {
    const int span = h->n * span_mult;
    if (h->drift_valid && h->drift_pc == p->pseudocount && h->drift_alen == p->alphabet_size && h->drift_span >= span) return GIBBS_OK;
    CUDA_TRY(h->pvals.reserve((size_t)span));
    pvals_kernel<<<(span + 255) / 256, 256, 0, h->stream>>>(span, p->pseudocount, ppm_den(h->n, p), h->pvals.p);
    CUDA_TRY(cudaGetLastError());
    if (launches) *launches += 1;
    int32_t rc = ensure_seq_counts(h, launches);
    if (rc) return rc;
    std::vector<int32_t> bc((size_t)h->n * 4);
    CUDA_TRY(cudaMemcpyAsync(bc.data(), h->basecnt.p, bc.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    long long g[4] = {0, 0, 0, 0};
    for (int32_t i = 0; i < h->n; ++i)
        for (int b = 0; b < 4; ++b) g[b] += bc[(size_t)i * 4 + b];
    for (int b = 0; b < 4; ++b) {
        if (g[b] > INT32_MAX) return fail(GIBBS_ERR_ARG, "more than 2^31 bases of one kind: background counts overflow int32 (the reference counts in int32, fs:34)");
        h->gcnt[b] = (int32_t)g[b];
    }
    h->drift_pc = p->pseudocount;
    h->drift_alen = p->alphabet_size;
    h->drift_span = span;
    h->drift_valid = true;
    return GIBBS_OK;
}

BgTables bg_tables(const gibbs_handle *h) {
    BgTables b;
    b.g = h->bg_g.p;
    b.gsum = h->bg_sum.p;
    b.gmax = h->bg_max.p;
    b.gmax_i = h->bg_max_i.p;
    b.wstride = h->bg_wstride;
    return b;
}

DeviceSeqs dev_seqs(const gibbs_handle *h) {
    DeviceSeqs s;
    s.packed = h->packed.p;
    s.len = h->len.p;
    s.n = h->n;
    s.row_words = h->row_words;
    s.uniform_len = h->min_len == h->max_len ? h->max_len : 0;
    s.mask = h->n_masked > 0 ? h->mask.p : nullptr;
    s.rowflag = h->n_masked > 0 ? h->rowflag.p : nullptr;
    s.wide = h->wide_valid ? h->wide.p : nullptr;
    s.wide_words = h->wide_words;
    return s;
}

int32_t upload(gibbs_handle *h, const uint8_t *seqs, const int64_t *offsets, int32_t n_seqs) {
    if (!seqs || !offsets) return fail(GIBBS_ERR_ARG, "null sequence buffer (ArgumentNullException)");
    if (n_seqs < 1) return fail(GIBBS_ERR_ARG, "n_seqs must be >= 1");
    int64_t max_len = 0, min_len = INT64_MAX;
    for (int32_t i = 0; i < n_seqs; ++i) {
        const int64_t l = offsets[i + 1] - offsets[i];
        if (l < 0) return fail(GIBBS_ERR_ARG, "offsets must be non-decreasing");
        if (l > max_len) max_len = l;
        if (l < min_len) min_len = l;
    }
    if (max_len > GIBBS_MAX_LEN) return fail(GIBBS_ERR_ARG, "sequence longer than %d", GIBBS_MAX_LEN);
    if (max_len < 1) return fail(GIBBS_ERR_SHORT_SEQ, "all sequences are empty");
    int32_t rc = set_device(h);
    if (rc) return rc;
    // whatever the handle held is gone from here on: a failure below must not leave the old n beside new buffers
    h->n = 0;
    h->start_chains = 0;
    h->run_done = false;
    h->wtab_valid = h->bg_valid = h->drift_valid = h->ss_valid = h->wide_valid = false;
    const int64_t total = offsets[n_seqs] - offsets[0];
    const int row_words = (int)(((max_len + 15) / 16 + 4 + 3) / 4 * 4);
    if (team_smem_bytes(row_words, 1) > 200 * 1024) return fail(GIBBS_ERR_ARG, "sequence too long for shared-memory staging");
    CUDA_TRY(h->ascii.reserve((size_t)(total > 0 ? total : 1)));
    CUDA_TRY(h->off.reserve((size_t)n_seqs + 1));
    CUDA_TRY(h->packed.reserve((size_t)n_seqs * row_words));
    CUDA_TRY(h->mask.reserve((size_t)n_seqs * row_words));
    CUDA_TRY(h->rowflag.reserve((size_t)n_seqs));
    CUDA_TRY(h->len.reserve((size_t)n_seqs));
    CUDA_TRY(h->flags.reserve(8));
    CUDA_TRY(h->symflags.reserve(4));
    std::vector<int64_t> rel((size_t)n_seqs + 1);
    for (int32_t i = 0; i <= n_seqs; ++i) rel[i] = offsets[i] - offsets[0];
    CUDA_TRY(cudaMemcpyAsync(h->ascii.p, seqs + offsets[0], (size_t)total, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemcpyAsync(h->off.p, rel.data(), rel.size() * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->flags.p, 0, 8 * sizeof(int), h->stream));
    CUDA_TRY(cudaMemsetAsync(h->symflags.p, 0, 4 * sizeof(int), h->stream));
    CUDA_TRY(cudaMemsetAsync(h->rowflag.p, 0, (size_t)n_seqs * sizeof(int32_t), h->stream));
    const int64_t words = (int64_t)n_seqs * row_words;
    pack_kernel<<<(unsigned)((words + 255) / 256), 256, 0, h->stream>>>(h->ascii.p, h->off.p, n_seqs, row_words, h->packed.p,
                                                                       h->mask.p, h->rowflag.p, h->len.p, h->symflags.p);
    CUDA_TRY(cudaGetLastError());
    int sym[4] = {0, 0, 0, 0};
    CUDA_TRY(cudaMemcpyAsync(sym, h->symflags.p, sizeof sym, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream)); // also keeps `rel` alive until the copy is done
    const int bad = sym[0];
    if (bad)
        return fail(GIBBS_ERR_SYMBOL, "symbol '%c' (0x%02x) is outside '*'..'Z', the range of the 49-slot tables "
                                      "(IndexOutOfRangeException, fs:17-20)",
                    (bad - 1) >= 32 && (bad - 1) < 127 ? (char)(bad - 1) : '?', bad - 1);
    h->n_masked = sym[1];
    h->has_gap = sym[2] != 0;
    h->n_gap = sym[2];
    try {
        h->len_host.resize((size_t)n_seqs);
    } catch (...) {
        return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    }
    for (int32_t i = 0; i < n_seqs; ++i) h->len_host[i] = (int32_t)(offsets[i + 1] - offsets[i]);
    h->n = n_seqs;
    h->row_words = row_words;
    h->max_len = (int32_t)max_len;
    h->min_len = (int32_t)min_len;
    return GIBBS_OK;
}

int32_t stage_sites(gibbs_handle *h, const int32_t *sites, int32_t heldout, int32_t k) {
    if (!sites) return fail(GIBBS_ERR_ARG, "null sites");
    if (heldout < -1 || heldout >= h->n) return fail(GIBBS_ERR_ARG, "heldout %d outside 0..%d", heldout, h->n - 1);
    // positions must address a full k-mer (getSegment, fs:149-153)
    CUDA_TRY(h->prim_sites.reserve((size_t)h->n));
    for (int32_t i = 0; i < h->n; ++i)
        if (i != heldout && sites[i] >= 0 && sites[i] + k > h->len_host[i])
            return fail(GIBBS_ERR_ARG, "site %d of sequence %d leaves the sequence (length %d, k %d)", sites[i], i, h->len_host[i], k);
    CUDA_TRY(cudaMemcpyAsync(h->prim_sites.p, sites, (size_t)h->n * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    return GIBBS_OK;
}

// the statistics of a run: its device counters (ST_* slots) and what the host recorded when it launched the run
void fill_stats(gibbs_run_stats *out, const unsigned long long *st, int launches, int fast, int team, int init_path, float ms) {
    out->site_updates = (int64_t)st[ST_SITE_UPDATES];
    out->window_scores = (int64_t)st[ST_WINDOW_SCORES];
    out->sweeps = (int64_t)st[ST_SWEEPS];
    out->exact_rescans = (int64_t)st[ST_EXACT_RESCANS];
    out->capped_chains = (int64_t)st[ST_CAPPED];
    out->speculative_discards = (int64_t)st[ST_SPECULATED];
    out->kernel_launches = launches;
    out->fast_path = fast;
    out->team_warps = team;
    out->init_path = init_path;
    out->kernel_ms = (double)ms;
}

// copies host to the device array dev when it differs from what was uploaded last (cache)
template <typename T>
int32_t upload_if_changed(std::vector<T> &host, std::vector<T> &cache, DevBuf<T> &dev, cudaStream_t stream) {
    if (host.size() * sizeof(T) != cache.size() * sizeof(T) || memcmp(host.data(), cache.data(), host.size() * sizeof(T)) != 0) {
        CUDA_TRY(dev.reserve(host.size()));
        CUDA_TRY(cudaMemcpyAsync(dev.p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice, stream));
        cache.swap(host);
    }
    return GIBBS_OK;
}

// Waits for the copies queued on h's stream, then reports a roulette pick of the last run that lay beyond the accumulated
// mass (MotifSampler: one error flag per set, S of them). A batch names the first such set by its number in the caller's
// list, set_base + s; a single-set handle passes set_base = -1 and names none.
int32_t sync_roulette(const gibbs_handle *h, int32_t S, int32_t set_base) {
    std::vector<int32_t> err;
    if (h->run_sampler == GIBBS_MOTIF_SAMPLER) {
        try {
            err.assign((size_t)S, 0);
        } catch (...) {
            return fail(GIBBS_ERR_NOMEM, "host allocation failed");
        }
        CUDA_TRY(cudaMemcpyAsync(err.data(), h->err_flag.p, (size_t)S * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    for (int32_t s = 0; s < (int32_t)err.size(); ++s) {
        if (!err[s]) continue;
        if (set_base < 0) return fail(GIBBS_ERR_ROULETTE, "a roulette pick lay beyond the accumulated mass (ArgumentException, fs:753)");
        return fail(GIBBS_ERR_ROULETTE, "set %d: a roulette pick lay beyond the accumulated mass (ArgumentException, fs:753)", set_base + s);
    }
    return GIBBS_OK;
}

// The winner of the promote-or-restart loop (fs:435-459) of each of the S sets of h's last run -- set s holds sequences
// seq_off[s] .. seq_off[s + 1] - 1 of the handle; a single-set handle is S = 1, seq_off {0, n} -- and what the fetch_best
// calls return of it. select(sites, m, motif, best_out, win_sums) launches the restart selection over the run's site
// entries into win_sites / win_scores; counts(sites, out) the PWM counts [S][k][4] of S site arrays. Everything is queued
// before the one synchronisation. st receives the run's device counters and extra_launches the launches made here, for
// the caller's statistics; set_base as in sync_roulette.
template <typename Select, typename Counts>
int32_t fetch_winners(gibbs_handle *h, int32_t S, const int32_t *seq_off, int32_t set_base, Select select, Counts counts,
                      int32_t *sites_out, double *scores_out, int32_t *n_out, double *sum_out, int32_t *restart_out,
                      int32_t *counts_out, unsigned long long *st, int *extra_launches) {
    const int32_t NT = h->n, M = h->run_m, k = h->run_k;
    const bool motif = h->run_sampler == GIBBS_MOTIF_SAMPLER;
    const size_t NS = (size_t)M * NT, per = (size_t)S * k * 4; // NS site entries of the winners (Positions lists for m = 2)
    std::vector<int32_t> best, pairs, counts2; // motifAmount = 2: the Positions lists and the counts of both their elements
    try {
        best.resize((size_t)S);
        if (sites_out && M == 2) pairs.resize(NS);
        if (counts_out && M == 2) counts2.resize(per * 2);
    } catch (...) {
        return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    }
    CUDA_TRY(h->win_sites.reserve(NS + S + (M == 2 ? 2 * (size_t)NT : 0)));
    CUDA_TRY(h->win_scores.reserve((size_t)NT + S));
    int32_t rc = select(M == 2 ? h->pos2.p : h->sites.p, M, motif ? 1 : 0, h->win_sites.p + NS, h->win_scores.p + NT);
    if (rc) return rc;
    *extra_launches = 1;
    CUDA_TRY(cudaMemcpyAsync(best.data(), h->win_sites.p + NS, (size_t)S * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (sum_out) CUDA_TRY(cudaMemcpyAsync(sum_out, h->win_scores.p + NT, (size_t)S * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (sites_out) // (motifAmount = 2: sites_out gets the newest position of each Positions list)
        CUDA_TRY(cudaMemcpyAsync(M == 1 ? sites_out : pairs.data(), h->win_sites.p, NS * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (scores_out) CUDA_TRY(cudaMemcpyAsync(scores_out, h->win_scores.p, (size_t)NT * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (counts_out) { // PWM counts of every winner's sites (all zero where the initial value survived: its sites are -1)
        CUDA_TRY(h->counts.reserve(per * M));
        for (int which = 0; which < M; ++which) { // motifAmount = 2: both elements of every Positions pair
            const int32_t *src = h->win_sites.p;
            if (M == 2) {
                int32_t *tmp = h->win_sites.p + NS + S + (size_t)which * NT;
                pair_element_kernel<<<(NT + 255) / 256, 256, 0, h->stream>>>(h->win_sites.p, NT, which, tmp);
                CUDA_TRY(cudaGetLastError());
                ++*extra_launches;
                src = tmp;
            }
            rc = counts(src, h->counts.p + per * which);
            if (rc) return rc;
            ++*extra_launches;
        }
        CUDA_TRY(cudaMemcpyAsync(M == 1 ? counts_out : counts2.data(), h->counts.p, per * M * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    }
    CUDA_TRY(cudaMemcpyAsync(st, h->stats.p, ST_NSLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    rc = sync_roulette(h, S, set_base);
    if (rc) return rc;
    h->best_valid = true;
    if (sites_out && M == 2)
        for (int32_t i = 0; i < NT; ++i) sites_out[i] = pairs[(size_t)2 * i];
    if (counts_out && M == 2)
        for (size_t e = 0; e < per; ++e) counts_out[e] = counts2[e] + counts2[per + e];
    for (int32_t s = 0; s < S; ++s) {
        // loop 0 [||] [|(0., 0)|] returned its initial value (quirk A.6-8); the MotifSampler's is [|{PWMS 0; Positions []}|]
        const bool initial = best[s] < 0;
        if (initial && sites_out) sites_out[seq_off[s]] = motif ? -1 : 0;
        if (initial && scores_out) scores_out[seq_off[s]] = 0.0;
        if (n_out) n_out[s] = initial ? 1 : seq_off[s + 1] - seq_off[s];
        if (restart_out) restart_out[s] = best[s];
    }
    return GIBBS_OK;
}

// MotifIndex.Positions of every restart of the last run (gibbs_fetch_positions, gibbs_batch_fetch_positions); missing is
// the message when there is no run
int32_t fetch_positions(gibbs_handle *h, int32_t m, int32_t *positions_out, const char *missing) {
    if (!h->run_done) return fail(GIBBS_ERR_ARG, "%s", missing);
    if (m != h->run_m) return fail(GIBBS_ERR_ARG, "the last run had motif_amount = %d", h->run_m);
    int32_t rc = set_device(h);
    if (rc) return rc;
    const size_t cells = (size_t)h->run_chains * h->n;
    CUDA_TRY(cudaMemcpyAsync(positions_out, m == 2 ? h->pos2.p : h->sites.p, cells * m * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return GIBBS_OK;
}

// the winners' Positions lists of the last fetch_best (gibbs_fetch_best_positions, gibbs_batch_fetch_best_positions);
// missing is the message when there is none
int32_t fetch_best_positions(gibbs_handle *h, int32_t m, int32_t *positions_out, const char *missing) {
    if (!h->run_done || !h->best_valid) return fail(GIBBS_ERR_ARG, "%s", missing);
    if (m != h->run_m) return fail(GIBBS_ERR_ARG, "the last run had motif_amount = %d", h->run_m);
    int32_t rc = set_device(h);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(positions_out, h->win_sites.p, (size_t)h->n * m * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return GIBBS_OK;
}

} // namespace

extern "C" {

int32_t gibbs_abi_version(void) { return GIBBS_ABI_VERSION; }

const char *gibbs_last_error(void) { return g_err; }

int32_t gibbs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int32_t gibbs_create(const uint8_t *seqs, const int64_t *offsets, int32_t n_seqs, int32_t device, gibbs_handle **out) {
    if (!out) return fail(GIBBS_ERR_ARG, "null out pointer");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1) {
        cudaGetLastError();
        return fail(GIBBS_ERR_CUDA, "no CUDA device available (%s); libgibbs_b200 has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    }
    if (device < 0 || device >= ndev) return fail(GIBBS_ERR_ARG, "device %d outside 0..%d", device, ndev - 1);
    gibbs_handle *h = new (std::nothrow) gibbs_handle();
    if (!h) return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    h->device = device;
    int32_t rc = set_device(h);
    if (!rc) {
        cudaError_t e2 = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
        if (e2 == cudaSuccess) e2 = cudaEventCreate(&h->ev0);
        if (e2 == cudaSuccess) e2 = cudaEventCreate(&h->ev1);
        if (e2 != cudaSuccess) rc = fail(GIBBS_ERR_CUDA, "stream/event creation: %s", cudaGetErrorString(e2));
        h->own_stream = true;
    }
    if (!rc) {
        cudaError_t e3 = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
        int optin = 0;
        if (e3 == cudaSuccess) e3 = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
        if (e3 != cudaSuccess) rc = fail(GIBBS_ERR_CUDA, "device attribute: %s", cudaGetErrorString(e3));
        h->smem_optin = (size_t)(optin > 0 ? optin : 0);
    }
    if (!rc) rc = upload(h, seqs, offsets, n_seqs);
    if (rc) {
        gibbs_destroy(h);
        return rc;
    }
    *out = h;
    return GIBBS_OK;
}

int32_t gibbs_upload(gibbs_handle *h, const uint8_t *seqs, const int64_t *offsets, int32_t n_seqs) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    return upload(h, seqs, offsets, n_seqs);
}

int32_t gibbs_destroy(gibbs_handle *h) {
    if (!h) return GIBBS_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h; // the device buffers, on the handle's device
    return GIBBS_OK;
}

int32_t gibbs_set_stream(gibbs_handle *h, void *cuda_stream) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    int32_t rc = set_device(h);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    if (cuda_stream) {
        h->stream = (cudaStream_t)cuda_stream;
        h->own_stream = false;
    } else {
        CUDA_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        h->own_stream = true;
    }
    return GIBBS_OK;
}

int32_t gibbs_num_sequences(const gibbs_handle *h) { return h ? h->n : 0; }

int32_t gibbs_set_team_warps(gibbs_handle *h, int32_t warps) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    if (warps != 0 && warps != 1 && warps != 4 && warps != 8 && warps != 16)
        return fail(GIBBS_ERR_ARG, "team size must be 0 (auto), 1, 4, 8 or 16 warps per chain");
    h->team_warps = warps;
    return GIBBS_OK;
}

int32_t gibbs_synchronize(gibbs_handle *h) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    int32_t rc = set_device(h);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return GIBBS_OK;
}

int32_t gibbs_loo_counts(gibbs_handle *h, const int32_t *sites, int32_t heldout, int32_t k, int32_t *counts_out) {
    if (!h || !counts_out) return fail(GIBBS_ERR_ARG, "null argument");
    if (h->n < 1) return fail(GIBBS_ERR_ARG, "handle holds no sequences");
    if (k < 1 || k > GIBBS_MAX_K) return fail(GIBBS_ERR_ARG, "motif width k=%d outside 1..%d", k, GIBBS_MAX_K);
    if (h->min_len < k) return fail(GIBBS_ERR_SHORT_SEQ, "a sequence of length %d is shorter than k=%d", h->min_len, k);
    int32_t rc = set_device(h);
    if (rc) return rc;
    rc = stage_sites(h, sites, heldout, k);
    if (rc) return rc;
    CUDA_TRY(h->prim_i32.reserve(GIBBS_MAX_K * 4 + 8));
    PrimArgs a{};
    a.s = dev_seqs(h);
    a.sites = h->prim_sites.p;
    a.heldout = heldout;
    a.k = k;
    a.counts_out = h->prim_i32.p;
    rc = launch_loo_counts(h, a);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(counts_out, h->prim_i32.p, (size_t)k * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return GIBBS_OK;
}

static int32_t scan_common(gibbs_handle *h, const int32_t *sites, int32_t heldout, const gibbs_params *p, int mode,
                           double *raw_out, double *log2_out, double *score_out, int32_t *site_out) {
    int32_t rc = check_params(h, p);
    if (rc) return rc;
    if (p->background != GIBBS_BG_FIXED) return fail(GIBBS_ERR_UNSUPPORTED, "the scan primitives take a fixed background (WithBPV)");
    if (heldout < 0 || heldout >= h->n) return fail(GIBBS_ERR_ARG, "heldout %d outside 0..%d", heldout, h->n - 1);
    rc = set_device(h);
    if (rc) return rc;
    rc = stage_sites(h, sites, heldout, p->k);
    if (rc) return rc;
    rc = ensure_wtab(h, p, nullptr);
    if (rc) return rc;
    const int W = h->len_host[heldout] - p->k + 1;
    CUDA_TRY(h->prim_f64.reserve((size_t)2 * W + 8));
    CUDA_TRY(h->prim_i32.reserve(GIBBS_MAX_K * 4 + 8));
    PrimArgs a{};
    a.s = dev_seqs(h);
    a.wtab = h->wtab.p;
    a.sites = h->prim_sites.p;
    a.heldout = heldout;
    a.k = p->k;
    a.fast_ok = fast_path_ok(h, p->k);
    a.raw_out = h->prim_f64.p;
    a.log2_out = h->prim_f64.p + W;
    a.score_out = h->prim_f64.p + 2 * (size_t)W;
    a.site_out = h->prim_i32.p;
    rc = launch_scan(h, a, mode);
    if (rc) return rc;
    if (mode == 0) {
        if (raw_out) CUDA_TRY(cudaMemcpyAsync(raw_out, a.raw_out, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (log2_out) CUDA_TRY(cudaMemcpyAsync(log2_out, a.log2_out, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    } else {
        if (score_out) CUDA_TRY(cudaMemcpyAsync(score_out, a.score_out, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (site_out) CUDA_TRY(cudaMemcpyAsync(site_out, a.site_out, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    }
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return GIBBS_OK;
}

int32_t gibbs_window_scores(gibbs_handle *h, const int32_t *sites, int32_t heldout, const gibbs_params *p, double *raw_out,
                            double *log2_out) {
    return scan_common(h, sites, heldout, p, 0, raw_out, log2_out, nullptr, nullptr);
}

int32_t gibbs_pick_argmax(gibbs_handle *h, const int32_t *sites, int32_t heldout, const gibbs_params *p, double *score_out,
                          int32_t *site_out) {
    return scan_common(h, sites, heldout, p, 1, nullptr, nullptr, score_out, site_out);
}

int32_t gibbs_pick_roulette(gibbs_handle *h, const int32_t *sites, int32_t heldout, const gibbs_params *p, double u,
                            double *pwms_out, int32_t *site_out) {
    int32_t rc = check_params(h, p);
    if (rc) return rc;
    if (p->background != GIBBS_BG_FIXED) return fail(GIBBS_ERR_UNSUPPORTED, "gibbs_pick_roulette takes a fixed background (WithPCV)");
    if (heldout < 0 || heldout >= h->n) return fail(GIBBS_ERR_ARG, "heldout %d outside 0..%d", heldout, h->n - 1);
    rc = set_device(h);
    if (rc) return rc;
    rc = stage_sites(h, sites, heldout, p->k);
    if (rc) return rc;
    rc = ensure_wtab(h, p, nullptr);
    if (rc) return rc;
    rc = ensure_bgtab(h, p, nullptr);
    if (rc) return rc;
    CUDA_TRY(h->cand_l.reserve((size_t)h->bg_wstride));
    CUDA_TRY(h->cand_w.reserve((size_t)h->bg_wstride));
    CUDA_TRY(h->prim_f64.reserve(8));
    CUDA_TRY(h->prim_i32.reserve(GIBBS_MAX_K * 4 + 8));
    RouletteArgs r{};
    r.p.s = dev_seqs(h);
    r.p.wtab = h->wtab.p;
    r.p.sites = h->prim_sites.p;
    r.p.heldout = heldout;
    r.p.k = p->k;
    r.p.fast_ok = fast_path_ok(h, p->k);
    r.bg = bg_tables(h);
    r.cutoff = p->cutoff;
    r.u = u;
    r.cand_l = h->cand_l.p;
    r.cand_w = h->cand_w.p;
    r.pwms_out = h->prim_f64.p;
    r.site_out = h->prim_i32.p;
    rc = launch_roulette(h, r);
    if (rc) return rc;
    double pw = 0.0;
    int32_t so[2] = {0, 0};
    CUDA_TRY(cudaMemcpyAsync(&pw, r.pwms_out, sizeof pw, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaMemcpyAsync(so, r.site_out, sizeof so, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    if (!so[1]) return fail(GIBBS_ERR_ROULETTE, "roulette pick %.17g lies beyond the accumulated mass (ArgumentException, fs:753)", u);
    if (pwms_out) *pwms_out = pw;
    if (site_out) *site_out = so[0];
    return GIBBS_OK;
}

int32_t gibbs_run_device(gibbs_handle *h, const gibbs_params *p, int32_t n_chains, int64_t chain_id_base, uint64_t seed,
                         int32_t rng_mode, const double *uniforms, int64_t uniforms_per_chain) {
    int32_t rc = check_params(h, p);
    if (rc) return rc;
    if (n_chains < 1) return fail(GIBBS_ERR_ARG, "n_chains must be >= 1");
    if (p->sampler != GIBBS_SITE_SAMPLER && p->sampler != GIBBS_MOTIF_SAMPLER) return fail(GIBBS_ERR_ARG, "unknown sampler %d", p->sampler);
    if (rng_mode != GIBBS_RNG_PHILOX && rng_mode != GIBBS_RNG_INJECTED) return fail(GIBBS_ERR_ARG, "unknown rng_mode %d", rng_mode);
    if (rng_mode == GIBBS_RNG_INJECTED && (!uniforms || uniforms_per_chain < 0)) return fail(GIBBS_ERR_ARG, "injected uniforms missing");
    const int m_amount = p->motif_amount <= 1 ? 1 : p->motif_amount;
    if (p->sampler == GIBBS_SITE_SAMPLER && m_amount != 1) return fail(GIBBS_ERR_ARG, "motif_amount belongs to the MotifSampler");
    if (m_amount > 2)
        return fail(GIBBS_ERR_UNSUPPORTED, "motifAmount = %d: combinations of one and two windows are built (fs:727-742); three and "
                                           "more sites per sequence are not", m_amount);
    if (h->n_masked > 0 && p->sampler != GIBBS_SITE_SAMPLER && m_amount != 1)
        return fail(GIBBS_ERR_UNSUPPORTED, "symbols outside A,C,G,T under the MotifSampler are built for motifAmount = 1 (motifAmount = 2 "
                                           "needs ACGT-only sequences)");
    rc = set_device(h);
    if (rc) return rc;
    h->run_done = false;
    int launches = 0;
    if (p->background == GIBBS_BG_FIXED) rc = ensure_wtab(h, p, &launches, m_amount);
    else rc = ensure_drift(h, p, &launches, m_amount);
    if (rc) return rc;
    const size_t cells = (size_t)n_chains * h->n;
    CUDA_TRY(h->sites.reserve(cells));
    CUDA_TRY(h->hv.reserve(cells));
    CUDA_TRY(h->scores.reserve(cells));
    CUDA_TRY(h->sums.reserve((size_t)n_chains));
    CUDA_TRY(h->stats.reserve(ST_NSLOTS));
    CUDA_TRY(h->best.reserve(1 + GIBBS_MAX_K * 4));
    CUDA_TRY(cudaMemsetAsync(h->stats.p, 0, ST_NSLOTS * sizeof(unsigned long long), h->stream));
    ChainArgs a{};
    a.s = dev_seqs(h);
    a.wtab = h->wtab.p;
    a.k = p->k;
    a.max_sweeps = p->max_sweeps > 0 ? p->max_sweeps : 1000000;
    a.fast_ok = p->background == GIBBS_BG_FIXED ? fast_path_ok(h, p->k) : 0;
    if (h->opt_exact_scans) a.fast_ok = 0;
    a.sampler = p->sampler;
    const int site_phases = GIBBS_PHASE_INIT | GIBBS_PHASE_GREEDY | GIBBS_PHASE_LEFT | GIBBS_PHASE_RIGHT;
    const int motif_phases = GIBBS_PHASE_INIT | GIBBS_PHASE_STOCHASTIC | GIBBS_PHASE_MOTIF_GREEDY;
    if (p->sampler == GIBBS_SITE_SAMPLER) {
        a.phase_mask = p->phase_mask ? p->phase_mask
                                     : (GIBBS_PHASE_INIT | GIBBS_PHASE_GREEDY | (p->phase_shifts ? (GIBBS_PHASE_LEFT | GIBBS_PHASE_RIGHT) : 0));
        if (a.phase_mask & ~site_phases) return fail(GIBBS_ERR_ARG, "phase_mask 0x%x has phases that are not SiteSampler phases", a.phase_mask);
    } else {
        a.phase_mask = p->phase_mask ? p->phase_mask : motif_phases;
        if (a.phase_mask & ~motif_phases) return fail(GIBBS_ERR_ARG, "phase_mask 0x%x has phases that are not MotifSampler phases", a.phase_mask);
    }
    const int start_m = h->start_m;
    h->start_m = 0;
    if (!(a.phase_mask & GIBBS_PHASE_INIT)) {
        if (start_m > m_amount) return fail(GIBBS_ERR_ARG, "the start state holds Positions lists of %d sites, motif_amount = %d", start_m, m_amount);
        if (h->start_chains != n_chains)
            return fail(GIBBS_ERR_ARG, "phase_mask without GIBBS_PHASE_INIT needs gibbs_set_start_state for %d chains", n_chains);
        if (h->start_max_excess > -p->k) // getSegment -> Array.take on a start position that leaves its sequence (fs:149-153)
            return fail(GIBBS_ERR_SHORT_SEQ, "a start site lies within %d symbols of the end of its sequence: no room for k = %d "
                                             "(InvalidOperationException from Array.take, fs:152)", -h->start_max_excess, p->k);
    }
    h->start_chains = 0;
    if (rng_mode == GIBBS_RNG_INJECTED) { // a stream that is too short must not turn into silent u = 0 draws
        int64_t need = 0;
        if (a.phase_mask & GIBBS_PHASE_INIT) need = (int64_t)h->n * (h->n - 1);
        if (a.phase_mask & GIBBS_PHASE_STOCHASTIC) need = (int64_t)h->n * (h->n - 1) + h->n; // draw index of fs:851 follows the random starts
        if (uniforms_per_chain < need)
            return fail(GIBBS_ERR_ARG, "uniforms_per_chain = %lld, but the phases of this run consume draws up to index %lld "
                                       "(N(N-1) random starts, then N roulette picks)", (long long)uniforms_per_chain, (long long)need);
    }
    a.rng_mode = rng_mode;
    a.seed = seed;
    a.chain_id_base = chain_id_base;
    a.uniforms = nullptr;
    a.uniforms_per_chain = 0;
    if (rng_mode == GIBBS_RNG_INJECTED) {
        const size_t nu = (size_t)n_chains * (size_t)uniforms_per_chain;
        CUDA_TRY(h->uniforms.reserve(nu > 0 ? nu : 1));
        if (nu) CUDA_TRY(cudaMemcpyAsync(h->uniforms.p, uniforms, nu * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        a.uniforms = h->uniforms.p;
        a.uniforms_per_chain = uniforms_per_chain;
    }
    a.n_chains = n_chains;
    a.sites = h->sites.p;
    a.hv = h->hv.p;
    a.scores = h->scores.p;
    a.sums = h->sums.p;
    a.stats = h->stats.p;
    a.cutoff = p->cutoff;
    memcpy(a.bg, p->bg, sizeof a.bg);
    a.ppm_given = nullptr;
    if (h->start_ppm_k != 0) {
        if (p->background != GIBBS_BG_DATA)
            return fail(GIBBS_ERR_ARG, "a start PPM is set (gibbs_set_start_ppm) but the run uses a fixed background: the reference "
                                       "has the ...OfPPM / ...WithPPM functions in the data-derived family only (fs:644, fs:1028)");
        if (h->start_ppm_k != p->k) return fail(GIBBS_ERR_ARG, "the start PPM has %d columns, the run k = %d", h->start_ppm_k, p->k);
        if (h->has_gap && p->alphabet_size >= 5)
            return fail(GIBBS_ERR_UNSUPPORTED, "a start PPM has rows A,C,G,T only, and the sequences hold Gap '-', which alphabet_size = %d "
                                               "includes: its PPM row is missing", p->alphabet_size);
        a.ppm_given = h->start_ppm.p;
    }
    const bool drift = p->background == GIBBS_BG_DATA;
    if (drift) { // both samplers' random starts and the SiteSampler's scans (drift_tables / drift_pick)
        a.pvals = h->pvals.p;
        a.basecnt = h->basecnt.p;
        a.maskcnt = h->n_masked > 0 ? h->maskcnt.p : nullptr; // symbols outside A,C,G,T per sequence (background denominators)
        a.ss = h->ss_valid ? h->ss.p : nullptr;
        a.ss_stride = h->max_len + 2;
        memcpy(a.gcnt, h->gcnt, sizeof a.gcnt);
        if (p->alphabet_size >= 5 && gap_row_built(p)) { // Gap has a row of its own (else it is dead like N)
            if (h->n_gap > INT32_MAX) return fail(GIBBS_ERR_ARG, "more than 2^31 Gaps: background counts overflow int32 (the reference counts in int32, fs:34)");
            a.gap_total = (int32_t)h->n_gap;
        }
        a.alpha_pc = (double)p->alphabet_size * p->pseudocount; // float alphabet.Length * pseudoCount, fs:117
        a.pc = p->pseudocount;
        // gibbs_set_option(GIBBS_OPT_EXACT_SCANS): every window in float64
        a.drift_fast_ok = h->opt_exact_scans ? 0 : drift_fast_path_ok(h->gcnt, a.gap_total, h->max_len, h->n, p);
    }
    if (p->sampler == GIBBS_MOTIF_SAMPLER) {
        Stage stages[MAX_STAGES] = {};
        const int n_stages = plan_stages(h, a, drift, stages);
        size_t warps = 0; // warps that hold a scratch list at once, over the stages of the run (the lists are indexed by CTA)
        for (int st = 0; st < n_stages; ++st)
            warps = std::max(warps, (size_t)(st == 0 ? n_chains : stages[st - 1].pause_below) * (size_t)stages[st].team);
        if (!drift) {
            rc = ensure_bgtab(h, p, &launches);
            if (rc) return rc;
        } else {
            h->bg_valid = false; // the fixed-background tables are not used; only the window stride is
            h->bg_wstride = h->max_len - p->k + 1;
            if (h->n_masked > 0 && h->bg_wstride < 64) h->bg_wstride = 64; // the candidate scratch doubles as a 49-slot symbol-count table
            CUDA_TRY(h->gbuf.reserve(warps * h->bg_wstride));
        }
        CUDA_TRY(h->cand_l.reserve(warps * h->bg_wstride)); // one scratch list per warp
        CUDA_TRY(h->cand_w.reserve(warps * h->bg_wstride));
        CUDA_TRY(h->err_flag.reserve(1));
        CUDA_TRY(cudaMemsetAsync(h->err_flag.p, 0, sizeof(int32_t), h->stream));
        MotifArgs m{};
        m.c = a;
        m.bg = bg_tables(h);
        m.cand_l = h->cand_l.p;
        m.cand_w = h->cand_w.p;
        m.error = h->err_flag.p;
        m.ascii = h->ascii.p;
        m.off = h->off.p;
        m.data_bg = drift ? 1 : 0;
        // the range check of the W table (ensure_wtab) or of the PPM values (drift_fast_path_ok)
        m.greedy_fast_ok = drift ? a.drift_fast_ok : a.fast_ok;
        if (drift) {
            m.pvals = a.pvals;
            m.basecnt = a.basecnt;
            memcpy(m.gcnt, a.gcnt, sizeof m.gcnt);
            m.alpha_pc = a.alpha_pc;
            m.pc = a.pc;
            m.gbuf = h->gbuf.p;
        }
        m.roulette_scan_ok = h->opt_exact_scans ? 0 : 1; // GIBBS_OPT_EXACT_SCANS: sequential roulette walk
        if (m_amount == 2) { // up to two sites per sequence: Positions lists beside the one-site state
            CUDA_TRY(h->pos2.reserve(cells * 2));
            CUDA_TRY(h->sc2.reserve((size_t)n_chains * h->bg_wstride));
            if (!(a.phase_mask & GIBBS_PHASE_INIT) && start_m < 2) // one-site start state: Positions = [site]
                CUDA_TRY(launch_motif2_seed(h->sites.p, (long long)cells, h->pos2.p, h->stream));
        }
        CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
        h->run_extra_launches = 0;
        {   // the random starts are the SiteSampler's (fs:876, fs:993): run them grid-wide whenever a kernel fits
            const int before = m.c.phase_mask;
            rc = launch_random_starts(h, m.c, drift);
            if (rc) return rc;
            m.init_done = (before & GIBBS_PHASE_INIT) && !(m.c.phase_mask & GIBBS_PHASE_INIT);
        }
        if (m_amount == 2) {
            Motif2Args q{};
            q.m = m;
            q.pos2 = h->pos2.p;
            q.sc = h->sc2.p;
            CUDA_TRY(launch_motif2(q, n_chains, team_smem_bytes(h->row_words, 1), h->stream));
            h->run_team = 1;
        } else {
            rc = launch_motif(h, m, stages, n_stages);
            if (rc) return rc;
        }
    } else {
        // teams of warps, speculative rounds and the hand-over of chain_kernel
        if (drift) a.fast_ok = a.drift_fast_ok;
        CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
        rc = launch_chain(h, a, drift);
        if (rc) return rc;
    }
    launches += h->run_extra_launches;
    h->run_sampler = p->sampler;
    h->run_m = p->sampler == GIBBS_MOTIF_SAMPLER ? m_amount : 1;
    h->best_valid = false;
    CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
    ++launches;
    best_chain_kernel<<<1, 256, 0, h->stream>>>(h->sums.p, n_chains, h->best.p);
    CUDA_TRY(cudaGetLastError());
    ++launches;
    h->run_chains = n_chains;
    h->run_k = p->k;
    h->run_fast = a.fast_ok;
    h->run_launches = launches;
    h->run_done = true;
    return GIBBS_OK;
}

int32_t gibbs_set_start_ppm(gibbs_handle *h, const double *ppm, int32_t k) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    if (!ppm) {
        h->start_ppm_k = 0;
        return GIBBS_OK;
    }
    if (k < 1 || k > GIBBS_MAX_K) return fail(GIBBS_ERR_ARG, "motif width k=%d outside 1..%d", k, GIBBS_MAX_K);
    int32_t rc = set_device(h);
    if (rc) return rc;
    CUDA_TRY(h->start_ppm.reserve((size_t)GIBBS_MAX_K * 4));
    CUDA_TRY(cudaMemcpyAsync(h->start_ppm.p, ppm, (size_t)k * 4 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream)); // the caller's buffer is free on return
    h->start_ppm_k = k;
    return GIBBS_OK;
}

int32_t gibbs_set_start_state(gibbs_handle *h, int32_t n_chains, const int32_t *sites, const double *scores) {
    if (!h || !sites || !scores) return fail(GIBBS_ERR_ARG, "null argument (ArgumentNullException)");
    if (h->n < 1 || n_chains < 1) return fail(GIBBS_ERR_ARG, "nothing to set");
    int32_t rc = set_device(h);
    if (rc) return rc;
    const size_t cells = (size_t)n_chains * h->n;
    // k is not known yet: remember how close a site comes to the end of its sequence; gibbs_run_device requires
    // site + k <= length (getSegment -> Array.take throws otherwise, fs:149-153)
    int32_t excess = INT32_MIN;
    for (size_t c = 0; c < cells; ++c) {
        const int32_t l = h->len_host[c % (size_t)h->n];
        if (sites[c] < -1 || sites[c] >= l) return fail(GIBBS_ERR_ARG, "start site %d outside its sequence", sites[c]);
        if (sites[c] >= 0 && sites[c] - l > excess) excess = sites[c] - l;
    }
    h->start_max_excess = excess;
    CUDA_TRY(h->sites.reserve(cells));
    CUDA_TRY(h->hv.reserve(cells));
    CUDA_TRY(h->scores.reserve(cells));
    CUDA_TRY(cudaMemcpyAsync(h->sites.p, sites, cells * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemcpyAsync(h->scores.p, scores, cells * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->hv.p, 0xFF, cells * sizeof(double), h->stream)); // all-ones = NaN marker
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    h->start_chains = n_chains;
    h->start_m = 0; // (gibbs_set_start_motif_state raises it after staging the Positions lists)
    h->run_done = false;
    return GIBBS_OK;
}

int32_t gibbs_set_start_motif_state(gibbs_handle *h, int32_t n_chains, int32_t m, const int32_t *positions, const double *pwms) {
    if (!h || !positions || !pwms) return fail(GIBBS_ERR_ARG, "null argument (ArgumentNullException)");
    if (m < 1 || m > 2) return fail(GIBBS_ERR_UNSUPPORTED, "Positions lists of %d sites: one and two are built", m);
    if (h->n < 1 || n_chains < 1) return fail(GIBBS_ERR_ARG, "nothing to set");
    const size_t cells = (size_t)n_chains * h->n;
    std::vector<int32_t> newest;
    try {
        newest.resize(cells);
    } catch (...) {
        return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    }
    for (size_t c = 0; c < cells; ++c) newest[c] = positions[c * m];
    int32_t rc = gibbs_set_start_state(h, n_chains, newest.data(), pwms); // validates the newest positions, stages scores
    if (rc) return rc;
    if (m == 2) {
        int32_t excess = h->start_max_excess;
        const int32_t *second = positions;
        for (size_t c = 0; c < cells; ++c) {
            const int32_t p0 = second[2 * c], p1 = second[2 * c + 1], l = h->len_host[c % (size_t)h->n];
            if (p1 < -1 || p1 >= l || (p0 < 0 && p1 >= 0)) return fail(GIBBS_ERR_ARG, "bad Positions list (second position %d)", p1);
            if (p1 >= 0 && p1 - l > excess) excess = p1 - l;
        }
        h->start_max_excess = excess;
        CUDA_TRY(h->pos2.reserve(cells * 2));
        CUDA_TRY(cudaMemcpyAsync(h->pos2.p, positions, cells * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    h->start_m = m;
    return GIBBS_OK;
}

int32_t gibbs_fetch_positions(gibbs_handle *h, int32_t m, int32_t *positions_out) {
    if (!h || !positions_out) return fail(GIBBS_ERR_ARG, "null argument");
    return fetch_positions(h, m, positions_out, "gibbs_fetch_positions without a preceding gibbs_run_device");
}

int32_t gibbs_fetch_best_positions(gibbs_handle *h, int32_t m, int32_t *positions_out) {
    if (!h || !positions_out) return fail(GIBBS_ERR_ARG, "null argument");
    return fetch_best_positions(h, m, positions_out, "gibbs_fetch_best_positions without a preceding gibbs_fetch_best");
}

int32_t gibbs_fetch(gibbs_handle *h, int32_t *sites_out, double *scores_out, double *sums_out, int32_t *best_chain_out,
                    int32_t *counts_out, gibbs_run_stats *stats_out) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    if (!h->run_done) return fail(GIBBS_ERR_ARG, "gibbs_fetch without a preceding gibbs_run_device");
    int32_t rc = set_device(h);
    if (rc) return rc;
    const size_t cells = (size_t)h->run_chains * h->n;
    int32_t best = 0;
    CUDA_TRY(cudaMemcpyAsync(&best, h->best.p, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (sites_out) CUDA_TRY(cudaMemcpyAsync(sites_out, h->sites.p, cells * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (scores_out) CUDA_TRY(cudaMemcpyAsync(scores_out, h->scores.p, cells * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (sums_out) CUDA_TRY(cudaMemcpyAsync(sums_out, h->sums.p, (size_t)h->run_chains * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    unsigned long long st[ST_NSLOTS];
    CUDA_TRY(cudaMemcpyAsync(st, h->stats.p, sizeof st, cudaMemcpyDeviceToHost, h->stream));
    rc = sync_roulette(h, 1, -1);
    if (rc) return rc;
    int extra_launches = 0;
    if (counts_out) {
        rc = launch_all_counts(h, dev_seqs(h), h->sites.p + (size_t)best * h->n, h->run_k, h->best.p + 1);
        if (rc) return rc;
        ++extra_launches;
        CUDA_TRY(cudaMemcpyAsync(counts_out, h->best.p + 1, (size_t)h->run_k * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    if (best_chain_out) *best_chain_out = best;
    if (stats_out) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        fill_stats(stats_out, st, h->run_launches + extra_launches, h->run_fast, h->run_team, h->run_init_path, ms);
    }
    return GIBBS_OK;
}

int32_t gibbs_fetch_best(gibbs_handle *h, int32_t repetitions, int32_t *sites_out, double *scores_out, int32_t *n_out,
                         double *sum_out, int32_t *restart_out, int32_t *counts_out, gibbs_run_stats *stats_out) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    if (!h->run_done) return fail(GIBBS_ERR_ARG, "gibbs_fetch_best without a preceding gibbs_run_device");
    if (repetitions < 0) repetitions = 0;
    int32_t rc = set_device(h);
    if (rc) return rc;
    auto select = [&](const int32_t *sites, int m, int motif, int32_t *best_out, double *win_sum) -> int32_t {
        restart_select_kernel<<<1, 32, 0, h->stream>>>(h->sums.p, sites, h->scores.p, h->run_chains, h->n, m * h->n, repetitions, motif,
                                                      best_out, h->win_sites.p, h->win_scores.p, win_sum);
        CUDA_TRY(cudaGetLastError());
        return GIBBS_OK;
    };
    auto counts = [&](const int32_t *sites, int32_t *out) { return launch_all_counts(h, dev_seqs(h), sites, h->run_k, out); };
    const int32_t seq_off[2] = {0, h->n};
    unsigned long long st[ST_NSLOTS];
    int extra_launches = 0;
    rc = fetch_winners(h, 1, seq_off, -1, select, counts, sites_out, scores_out, n_out, sum_out, restart_out, counts_out, st,
                       &extra_launches);
    if (rc) return rc;
    if (stats_out) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        fill_stats(stats_out, st, h->run_launches + extra_launches, h->run_fast, h->run_team, h->run_init_path, ms);
    }
    return GIBBS_OK;
}

int32_t gibbs_set_option(gibbs_handle *h, int32_t option, int32_t value) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    switch (option) {
    case GIBBS_OPT_INIT_PATH:
        if (value < GIBBS_INIT_AUTO || value > GIBBS_INIT_TILED) return fail(GIBBS_ERR_ARG, "GIBBS_OPT_INIT_PATH takes GIBBS_INIT_AUTO .. GIBBS_INIT_TILED");
        h->opt_init_path = value;
        return GIBBS_OK;
    case GIBBS_OPT_EXACT_SCANS:
        h->opt_exact_scans = value != 0;
        return GIBBS_OK;
    case GIBBS_OPT_MIN_WIDTH:
        if (value < -1 || value > 128) return fail(GIBBS_ERR_ARG, "GIBBS_OPT_MIN_WIDTH takes -1 (automatic) .. 128");
        h->opt_min_width = value;
        return GIBBS_OK;
    case GIBBS_OPT_SEQ_SWEEPS:
        if (value < 0 || value > 3) return fail(GIBBS_ERR_ARG, "GIBBS_OPT_SEQ_SWEEPS takes 0 .. 3");
        h->opt_seq_sweeps = value;
        return GIBBS_OK;
    case GIBBS_OPT_TILE_ROWS:
        if (value < 0) return fail(GIBBS_ERR_ARG, "GIBBS_OPT_TILE_ROWS takes 0 (what fits) or a positive number of sequences");
        h->opt_tile_rows = value;
        return GIBBS_OK;
    case GIBBS_OPT_CLUSTER:
        if (value != 0 && value != 4 && value != 8) return fail(GIBBS_ERR_ARG, "GIBBS_OPT_CLUSTER takes 0, 4 or 8");
        h->opt_cluster = value;
        return GIBBS_OK;
    case GIBBS_OPT_STAGE2_AT:
    case GIBBS_OPT_STAGE3_AT:
        if (value < 1 || value > 16) return fail(GIBBS_ERR_ARG, "hand-over thresholds are 1 .. 16 chains per SM");
        (option == GIBBS_OPT_STAGE2_AT ? h->opt_stage2_at : h->opt_stage3_at) = value;
        if (h->opt_stage3_at > h->opt_stage2_at) h->opt_stage3_at = h->opt_stage2_at;
        return GIBBS_OK;
    default:
        return fail(GIBBS_ERR_ARG, "unknown option %d", option);
    }
}

int32_t gibbs_run(gibbs_handle *h, const gibbs_params *p, int32_t n_chains, int64_t chain_id_base, uint64_t seed,
                  int32_t rng_mode, const double *uniforms, int64_t uniforms_per_chain, int32_t *sites_out,
                  double *scores_out, double *sums_out, int32_t *best_chain_out, int32_t *counts_out,
                  gibbs_run_stats *stats_out) {
    int32_t rc = gibbs_run_device(h, p, n_chains, chain_id_base, seed, rng_mode, uniforms, uniforms_per_chain);
    if (rc) return rc;
    return gibbs_fetch(h, sites_out, scores_out, sums_out, best_chain_out, counts_out, stats_out);
}

/* ---- one process, several devices ------------------------------------------------------------------------------- */
struct gibbs_multi {
    std::vector<gibbs_handle *> dev;
    std::vector<int32_t> first, count; // chains [first, first + count) of the last run live on device i
    std::vector<double> sums;          // sums of every restart of the last run, in restart order
    int32_t run_chains = 0;
    bool run_done = false;
};

int32_t gibbs_multi_create(const uint8_t *seqs, const int64_t *offsets, int32_t n_seqs, const int32_t *devices,
                           int32_t n_devices, gibbs_multi **out) {
    if (!out) return fail(GIBBS_ERR_ARG, "null out pointer");
    *out = nullptr;
    const int32_t visible = gibbs_device_count();
    if (visible < 1) return fail(GIBBS_ERR_CUDA, "no CUDA device available; libgibbs_b200 has no CPU fallback");
    if (n_devices == 0) n_devices = visible; // 0 = every visible device
    // (an explicit device list may name a device twice: two slots then share it)
    if (n_devices < 1 || (!devices && n_devices > visible)) return fail(GIBBS_ERR_ARG, "n_devices = %d, %d visible", n_devices, visible);
    gibbs_multi *m = new (std::nothrow) gibbs_multi();
    if (!m) return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    for (int32_t i = 0; i < n_devices; ++i) {
        gibbs_handle *h = nullptr;
        const int32_t rc = gibbs_create(seqs, offsets, n_seqs, devices ? devices[i] : i, &h); // the set is replicated
        if (rc) {
            gibbs_multi_destroy(m);
            return rc;
        }
        m->dev.push_back(h);
    }
    m->first.assign((size_t)n_devices, 0);
    m->count.assign((size_t)n_devices, 0);
    *out = m;
    return GIBBS_OK;
}

int32_t gibbs_multi_destroy(gibbs_multi *m) {
    if (!m) return GIBBS_OK;
    for (gibbs_handle *h : m->dev) gibbs_destroy(h);
    delete m;
    return GIBBS_OK;
}

int32_t gibbs_multi_num_devices(const gibbs_multi *m) { return m ? (int32_t)m->dev.size() : 0; }

gibbs_handle *gibbs_multi_handle(gibbs_multi *m, int32_t i) {
    return (m && i >= 0 && i < (int32_t)m->dev.size()) ? m->dev[(size_t)i] : nullptr;
}

int32_t gibbs_multi_run_device(gibbs_multi *m, const gibbs_params *p, int32_t n_chains, int64_t chain_id_base, uint64_t seed,
                               int32_t rng_mode, const double *uniforms, int64_t uniforms_per_chain) {
    if (!m || m->dev.empty()) return fail(GIBBS_ERR_ARG, "null multi-device handle");
    if (n_chains < 1) return fail(GIBBS_ERR_ARG, "n_chains must be >= 1");
    m->run_done = false;
    const int32_t G = (int32_t)m->dev.size();
    // contiguous blocks of restarts per device; streams are keyed by the global chain id, so the result of every
    // restart is the one a single device would compute. Launches are asynchronous: the devices run concurrently.
    int32_t next = 0;
    for (int32_t i = 0; i < G; ++i) {
        const int32_t cnt = n_chains / G + (i < n_chains % G ? 1 : 0);
        m->first[(size_t)i] = next;
        m->count[(size_t)i] = cnt;
        if (cnt > 0) {
            const double *u = (rng_mode == GIBBS_RNG_INJECTED && uniforms) ? uniforms + (size_t)next * (size_t)uniforms_per_chain : uniforms;
            const int32_t rc = gibbs_run_device(m->dev[(size_t)i], p, cnt, chain_id_base + next, seed, rng_mode, u, uniforms_per_chain);
            if (rc) return rc;
        }
        next += cnt;
    }
    m->run_chains = n_chains;
    m->run_done = true;
    return GIBBS_OK;
}

namespace {
// rows of restart r (global index) of the last multi-device run
int32_t multi_rows(gibbs_multi *m, int32_t r, int32_t *sites_out, double *scores_out) {
    for (size_t i = 0; i < m->dev.size(); ++i) {
        if (r < m->first[i] || r >= m->first[i] + m->count[i]) continue;
        gibbs_handle *h = m->dev[i];
        int32_t rc = set_device(h);
        if (rc) return rc;
        const size_t o = (size_t)(r - m->first[i]) * h->n;
        if (sites_out) CUDA_TRY(cudaMemcpyAsync(sites_out, h->sites.p + o, (size_t)h->n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
        if (scores_out) CUDA_TRY(cudaMemcpyAsync(scores_out, h->scores.p + o, (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        return GIBBS_OK;
    }
    return fail(GIBBS_ERR_ARG, "restart %d is not part of the last run", r);
}
} // namespace

int32_t gibbs_multi_fetch_best(gibbs_multi *m, int32_t repetitions, int32_t *sites_out, double *scores_out, int32_t *n_out,
                               double *sum_out, int32_t *restart_out, int32_t *counts_out, gibbs_run_stats *stats_out) {
    if (!m || m->dev.empty()) return fail(GIBBS_ERR_ARG, "null multi-device handle");
    if (!m->run_done) return fail(GIBBS_ERR_ARG, "gibbs_multi_fetch_best without a preceding gibbs_multi_run_device");
    if (repetitions < 0) repetitions = 0;
    const int32_t N = m->dev[0]->n, R = m->run_chains;
    if (m->dev[0]->run_m != 1) return fail(GIBBS_ERR_UNSUPPORTED, "the multi-device calls return one site per sequence (motif_amount = 1)");
    try {
        m->sums.assign((size_t)R, 0.0);
    } catch (...) {
        return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    }
    gibbs_run_stats total{};
    for (size_t i = 0; i < m->dev.size(); ++i) { // 8 B per restart and the counters of each device: all that always crosses PCIe
        if (m->count[i] == 0) continue;
        gibbs_run_stats st{};
        const int32_t rc = gibbs_fetch(m->dev[i], nullptr, nullptr, m->sums.data() + m->first[i], nullptr, nullptr, &st);
        if (rc) return rc;
        total.site_updates += st.site_updates; total.window_scores += st.window_scores; total.sweeps += st.sweeps;
        total.exact_rescans += st.exact_rescans; total.capped_chains += st.capped_chains;
        total.speculative_discards += st.speculative_discards; total.kernel_launches += st.kernel_launches;
        total.fast_path = st.fast_path; total.team_warps = st.team_warps; total.init_path = st.init_path;
        if (st.kernel_ms > total.kernel_ms) total.kernel_ms = st.kernel_ms; // the devices ran concurrently
    }
    // the promote-or-restart loop of fs:435-459 (quirk A.6-8) over the restarts in their global order; see
    // restart_select_kernel for the single-device twin. `acc = best` needs the arrays only when two sums are equal.
    const bool motif = m->dev[0]->run_sampler == GIBBS_MOTIF_SAMPLER;
    std::vector<int32_t> sa, sb;
    std::vector<double> va, vb;
    int32_t best = -1, acc = -1, r = 0; // acc -1 = [||]
    double bsum = 0.0;
    for (long long n = 0; n <= (long long)repetitions; ++n) {
        if (acc >= 0 && m->sums[(size_t)acc] == bsum) { // acc = best ?
            bool same;
            try {
                sa.resize((size_t)N); va.resize((size_t)N);
                int32_t rc = multi_rows(m, acc, sa.data(), va.data());
                if (rc) return rc;
                if (best < 0) {
                    same = N == 1 && va[0] == 0.0 && sa[0] == (motif ? -1 : 0);
                } else {
                    sb.resize((size_t)N); vb.resize((size_t)N);
                    rc = multi_rows(m, best, sb.data(), vb.data());
                    if (rc) return rc;
                    same = true;
                    for (int32_t i = 0; i < N && same; ++i) same = sa[(size_t)i] == sb[(size_t)i] && va[(size_t)i] == vb[(size_t)i];
                }
            } catch (...) {
                return fail(GIBBS_ERR_NOMEM, "host allocation failed");
            }
            if (same) break;
        }
        const double asum = acc >= 0 ? m->sums[(size_t)acc] : 0.0;
        if (asum > bsum) { // promote (an empty acc leaves best as it is)
            if (acc >= 0) { best = acc; bsum = asum; }
            acc = -1;
        } else {
            if (r >= R) break; // (cannot happen with n_chains >= repetitions + 1)
            acc = r++;
        }
    }
    if (best >= 0) {
        const int32_t rc = multi_rows(m, best, sites_out, scores_out);
        if (rc) return rc;
        if (counts_out) {
            for (size_t i = 0; i < m->dev.size(); ++i) {
                if (best < m->first[i] || best >= m->first[i] + m->count[i]) continue;
                gibbs_handle *h = m->dev[i];
                int32_t rc2 = set_device(h);
                if (rc2) return rc2;
                rc2 = launch_all_counts(h, dev_seqs(h), h->sites.p + (size_t)(best - m->first[i]) * h->n, h->run_k, h->best.p + 1);
                if (rc2) return rc2;
                CUDA_TRY(cudaMemcpyAsync(counts_out, h->best.p + 1, (size_t)h->run_k * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
                CUDA_TRY(cudaStreamSynchronize(h->stream));
                total.kernel_launches += 1;
            }
        }
    } else {
        if (sites_out) sites_out[0] = motif ? -1 : 0;
        if (scores_out) scores_out[0] = 0.0;
        if (counts_out) memset(counts_out, 0, (size_t)m->dev[0]->run_k * 4 * sizeof(int32_t));
    }
    if (n_out) *n_out = best < 0 ? 1 : N;
    if (sum_out) *sum_out = best < 0 ? 0.0 : m->sums[(size_t)best];
    if (restart_out) *restart_out = best;
    if (stats_out) *stats_out = total;
    return GIBBS_OK;
}

int32_t gibbs_device_results(gibbs_handle *h, void **sites_dev, void **scores_dev, void **sums_dev) {
    if (!h) return fail(GIBBS_ERR_ARG, "null handle");
    if (!h->run_done) return fail(GIBBS_ERR_ARG, "no run on this handle yet");
    if (sites_dev) *sites_dev = h->sites.p;
    if (scores_dev) *scores_dev = h->scores.p;
    if (sums_dev) *sums_dev = h->sums.p;
    return GIBBS_OK;
}

int32_t gibbs_host_alloc(size_t bytes, void **ptr_out) {
    if (!ptr_out) return fail(GIBBS_ERR_ARG, "null output");
    *ptr_out = nullptr;
    if (bytes == 0) return GIBBS_OK;
    const cudaError_t e = cudaHostAlloc(ptr_out, bytes, cudaHostAllocPortable);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(GIBBS_ERR_NOMEM, "cudaHostAlloc of %zu bytes failed", bytes);
    }
    CUDA_TRY(e);
    return GIBBS_OK;
}

int32_t gibbs_host_free(void *ptr) {
    if (ptr) CUDA_TRY(cudaFreeHost(ptr));
    return GIBBS_OK;
}

int32_t gibbs_measure_smem_bandwidth(int32_t device, int32_t iters, double *gbps_out, double *ms_out) {
    if (!gbps_out) return fail(GIBBS_ERR_ARG, "null output");
    if (iters < 1) iters = 1;
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    unsigned int *sink = nullptr;
    CUDA_TRY(cudaMalloc(&sink, sizeof(unsigned int)));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int grid = prop.multiProcessorCount * 2;
    smem_stream_kernel<<<grid, 1024>>>(iters, sink); // warm-up
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
    float best_ms = 1e30f;
    for (int rep = 0; rep < 5; ++rep) {
        CUDA_TRY(cudaEventRecord(e0));
        smem_stream_kernel<<<grid, 1024>>>(iters, sink);
        CUDA_TRY(cudaEventRecord(e1));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        if (ms < best_ms) best_ms = ms;
    }
    const double bytes = (double)grid * 1024.0 * 16.0 * 8.0 * (double)iters;
    *gbps_out = bytes / ((double)best_ms * 1e-3) / 1e9;
    if (ms_out) *ms_out = (double)best_ms;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    return GIBBS_OK;
}

/* ---- many independent sequence sets in one launch ------------------------------------------------------------------ */
// The sets are uploaded as one concatenation into an internal handle (rows with a common row_words, lengths, mask plane,
// stream, events); every set then gets its own ChainArgs that point into it (gibbs_batch.cuh), and for the MotifSampler its
// own Motif2Args (gibbs_motif_batch.cuh). Per-set W / drift / background window tables are built with the single-set setup
// kernels, one small launch per set, and kept while the parameters stay the same. The run state, results and scratch are
// the internal handle's, set-major (set s at R seq_off[s], restart-major within it) with one roulette flag per set in
// err_flag; the handle's own table caches stay unset, since the batch keeps its tables per set.
struct gibbs_batch {
    gibbs_handle *h = nullptr;
    int32_t n_sets = 0, n_seqs = 0;
    // a block of a gibbs_multi_batch holds sets set_base .. set_base + n_sets - 1 of set_total: messages name sets by that
    // number and the chain-count limit applies to set_total (a batch of its own: 0 and n_sets)
    int32_t set_base = 0, set_total = 0;
    std::vector<int32_t> seq_off;               // [n_sets + 1] first sequence of each set
    std::vector<int32_t> min_len, max_len;      // per set
    std::vector<int64_t> n_masked;              // symbols outside A,C,G,T per set
    std::vector<int64_t> n_gap;                 // per set: Gaps '-'
    std::vector<int64_t> gcnt;                  // [n_sets][4] A,C,G,T counts (the data-derived background)
    DevBuf<int32_t> d_seq_off;
    // per-set tables, keyed by the parameters they were built for
    DevBuf<WEnt> wtab;                          // set s at 4 m seq_off[s]: counts 0 .. m N_s - 1 (m = motifAmount)
    DevBuf<int> wt_range;                       // [n_sets][4]: min lg, max lg, non-normal W
    DevBuf<double> pvals;                       // set s at m seq_off[s]
    std::vector<int32_t> fast;                  // per set: the fixed-point ranking pass is usable
    // MotifSampler, fixed background: background-only window tables (bg_setup_kernel), set s at g_off[s] with its own stride
    DevBuf<double> bg_g, bg_sum, bg_max;
    DevBuf<int32_t> bg_max_i;
    std::vector<size_t> g_off;
    bool tab_valid = false;
    int32_t tab_bgmode = -1, tab_alen = 0, tab_k = 0, tab_m = 0, tab_bgwin = 0;
    double tab_pc = 0;
    std::vector<double> tab_bg;
    // per-set arguments and launch groups (uploaded when they change)
    std::vector<ChainArgs> args_host;
    std::vector<Motif2Args> margs_host;
    std::vector<int32_t> groups_host;           // per group: set ids, then chain offsets
    DevBuf<ChainArgs> d_args;
    DevBuf<Motif2Args> d_margs;
    DevBuf<int32_t> d_groups;
};

namespace {

constexpr int BATCH_GROUPS = 4; // (masked symbols) x (4 warps per chain, 1 warp)

int batch_team(const gibbs_batch *b, int s) {
    const int N = b->seq_off[s + 1] - b->seq_off[s];
    return (N >= 4 && team_smem_bytes(b->h->row_words, 4) <= 200 * 1024) ? 4 : 1;
}

// motif: gibbs_batch_run_motif_device (the MotifSampler), else gibbs_batch_run_device (the SiteSampler)
int32_t batch_check(const gibbs_batch *b, const gibbs_params *p, const double *bg_per_set, int32_t R, bool motif) {
    if (!b) return fail(GIBBS_ERR_ARG, "null batch");
    if (!p) return fail(GIBBS_ERR_ARG, "null params");
    if (R < 1) return fail(GIBBS_ERR_ARG, "restarts_per_set must be >= 1");
    if (!motif) {
        if (p->sampler != GIBBS_SITE_SAMPLER)
            return fail(p->sampler == GIBBS_MOTIF_SAMPLER ? GIBBS_ERR_UNSUPPORTED : GIBBS_ERR_ARG,
                        "gibbs_batch_run_device runs the SiteSampler (sampler = %d); MotifSampler batches run in "
                        "gibbs_batch_run_motif_device", p->sampler);
        if (p->motif_amount > 1) return fail(GIBBS_ERR_ARG, "motif_amount belongs to the MotifSampler");
    } else {
        if (p->sampler != GIBBS_MOTIF_SAMPLER)
            return fail(GIBBS_ERR_ARG, "gibbs_batch_run_motif_device runs the MotifSampler (sampler = %d)", p->sampler);
        if (p->motif_amount > 2)
            return fail(GIBBS_ERR_UNSUPPORTED, "motifAmount = %d: combinations of one and two windows are built (fs:727-742); three "
                                               "and more sites per sequence are not", p->motif_amount);
    }
    if (p->phase_mask != 0) return fail(GIBBS_ERR_ARG, "batches run the whole pipeline: phase_mask must be 0");
    if (p->k < 1 || p->k > GIBBS_MAX_K) return fail(GIBBS_ERR_ARG, "motif width k=%d outside 1..%d", p->k, GIBBS_MAX_K);
    if (p->alphabet_size < 1) return fail(GIBBS_ERR_ARG, "alphabet_size must be >= 1");
    if (!(p->pseudocount >= 0.0)) return fail(GIBBS_ERR_ARG, "pseudocount must be >= 0");
    if (p->background != GIBBS_BG_FIXED && p->background != GIBBS_BG_DATA) return fail(GIBBS_ERR_ARG, "unknown background mode %d", p->background);
    if ((int64_t)R * b->set_total > INT32_MAX) return fail(GIBBS_ERR_ARG, "%d sets x %d restarts: too many chains", b->set_total, R);
    for (int32_t s = 0; s < b->n_sets; ++s) {
        const int32_t gs = b->set_base + s; // the set's number in the caller's list
        if (b->min_len[s] < p->k) {
            int32_t i = b->seq_off[s];
            while (b->h->len_host[i] >= p->k) ++i;
            return fail(GIBBS_ERR_SHORT_SEQ, "set %d, sequence %d: length %d is shorter than k=%d (Array.take, fs:152)", gs,
                        i - b->seq_off[s], b->h->len_host[i], p->k);
        }
        if (b->n_gap[s] > 0 && p->alphabet_size >= 5 && (motif || !gap_row_built(p)))
            return fail(GIBBS_ERR_UNSUPPORTED, "set %d holds Gap '-' and alphabet_size = %d includes it: its PWM row is built for the "
                                               "SiteSampler with the data-derived background only (pass alphabet_size = 4 to score Gap "
                                               "like any other non-alphabet symbol)", gs, p->alphabet_size);
        if (motif && p->motif_amount == 2 && b->n_masked[s] > 0)
            return fail(GIBBS_ERR_UNSUPPORTED, "set %d holds symbols outside A,C,G,T: the MotifSampler builds them for motifAmount = 1 "
                                               "(motifAmount = 2 needs ACGT-only sequences)", gs);
        const double *bg = p->background == GIBBS_BG_FIXED && bg_per_set ? bg_per_set + 4 * (size_t)s : p->bg;
        if (p->background == GIBBS_BG_FIXED)
            for (int x = 0; x < 4; ++x)
                if (!(bg[x] > 0.0)) return fail(GIBBS_ERR_ARG, "set %d: background probability bg[%d] must be > 0", gs, x);
        if (p->background == GIBBS_BG_DATA)
            for (int x = 0; x < 4; ++x)
                if (b->gcnt[4 * (size_t)s + x] > INT32_MAX || b->n_gap[s] > INT32_MAX)
                    return fail(GIBBS_ERR_ARG, "set %d: more than 2^31 bases of one kind: background counts overflow int32 (fs:34)", gs);
    }
    return GIBBS_OK;
}

// the Gap slot of set s's totals when Gap has a row of its own (checked against int32 in batch_check), else 0
int32_t batch_gap_total(const gibbs_batch *b, const gibbs_params *p, int32_t s) {
    return p->alphabet_size >= 5 && gap_row_built(p) ? (int32_t)b->n_gap[s] : 0;
}

DeviceSeqs batch_seqs(const gibbs_batch *b, int32_t s) {
    const gibbs_handle *h = b->h;
    const int32_t o = b->seq_off[s];
    DeviceSeqs d{};
    d.packed = h->packed.p + (size_t)o * h->row_words;
    d.len = h->len.p + o;
    d.n = b->seq_off[s + 1] - o;
    d.row_words = h->row_words;
    d.uniform_len = b->min_len[s] == b->max_len[s] ? b->max_len[s] : 0;
    d.mask = b->n_masked[s] > 0 ? h->mask.p + (size_t)o * h->row_words : nullptr;
    d.rowflag = b->n_masked[s] > 0 ? h->rowflag.p + o : nullptr;
    return d;
}

// Tables of every set, with the kernels of ensure_wtab / ensure_drift / ensure_bgtab: W tables (fixed background) or PPM
// value tables (data-derived) over m N_s counts (m = motifAmount; the denominator keeps N_s), and for the MotifSampler on
// the fixed background (bg_win) the background-only window tables
int32_t batch_tables(gibbs_batch *b, const gibbs_params *p, const double *bg_per_set, int m, bool bg_win, int *launches) {
    gibbs_handle *h = b->h;
    std::vector<double> bg((size_t)b->n_sets * 4);
    for (int32_t s = 0; s < b->n_sets; ++s)
        for (int x = 0; x < 4; ++x) bg[4 * (size_t)s + x] = bg_per_set ? bg_per_set[4 * (size_t)s + x] : p->bg[x];
    const bool fixed = p->background == GIBBS_BG_FIXED;
    if (b->tab_valid && b->tab_bgmode == p->background && b->tab_pc == p->pseudocount && b->tab_alen == p->alphabet_size &&
        b->tab_k == p->k && b->tab_m == m && b->tab_bgwin == (int)bg_win && (!fixed || b->tab_bg == bg))
        return GIBBS_OK;
    b->tab_valid = false;
    b->fast.assign((size_t)b->n_sets, 0);
    if (fixed) {
        CUDA_TRY(b->wtab.reserve((size_t)b->n_seqs * 4 * m));
        CUDA_TRY(b->wt_range.reserve((size_t)b->n_sets * 4));
        std::vector<int> range((size_t)b->n_sets * 4);
        for (int32_t s = 0; s < b->n_sets; ++s) {
            range[4 * (size_t)s] = INT32_MAX;
            range[4 * (size_t)s + 1] = INT32_MIN;
            range[4 * (size_t)s + 2] = range[4 * (size_t)s + 3] = 0;
        }
        CUDA_TRY(cudaMemcpyAsync(b->wt_range.p, range.data(), range.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        for (int32_t s = 0; s < b->n_sets; ++s) {
            const int N = b->seq_off[s + 1] - b->seq_off[s], span = N * m;
            const double *q = bg.data() + 4 * (size_t)s;
            wtab_kernel<<<(span * 4 + 255) / 256, 256, 0, h->stream>>>(span, p->pseudocount, ppm_den(N, p), q[0], q[1], q[2], q[3],
                                                                       b->wtab.p + 4 * (size_t)m * b->seq_off[s], b->wt_range.p + 4 * (size_t)s);
            CUDA_TRY(cudaGetLastError());
        }
        *launches += b->n_sets;
        if (bg_win) {
            b->g_off.assign((size_t)b->n_sets + 1, 0);
            for (int32_t s = 0; s < b->n_sets; ++s)
                b->g_off[s + 1] = b->g_off[s] + (size_t)(b->seq_off[s + 1] - b->seq_off[s]) * (size_t)(b->max_len[s] - p->k + 1);
            CUDA_TRY(b->bg_g.reserve(b->g_off[b->n_sets]));
            CUDA_TRY(b->bg_sum.reserve((size_t)b->n_seqs));
            CUDA_TRY(b->bg_max.reserve((size_t)b->n_seqs));
            CUDA_TRY(b->bg_max_i.reserve((size_t)b->n_seqs));
            for (int32_t s = 0; s < b->n_sets; ++s) {
                const int32_t o = b->seq_off[s], N = b->seq_off[s + 1] - o;
                const double *q = bg.data() + 4 * (size_t)s;
                bg_setup_kernel<<<(N + 127) / 128, 128, 0, h->stream>>>(batch_seqs(b, s), p->k, q[0], q[1], q[2], q[3], b->max_len[s] - p->k + 1,
                                                                       b->bg_g.p + b->g_off[s], b->bg_sum.p + o, b->bg_max.p + o, b->bg_max_i.p + o);
                CUDA_TRY(cudaGetLastError());
            }
            *launches += b->n_sets;
        }
        CUDA_TRY(cudaMemcpyAsync(range.data(), b->wt_range.p, range.size() * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        for (int32_t s = 0; s < b->n_sets; ++s)
            b->fast[s] = fast_path_ok_range(range[4 * (size_t)s + 2], range[4 * (size_t)s], range[4 * (size_t)s + 1], p->k);
    } else {
        // base counts, symbols outside A,C,G,T and prefix tables per sequence; the background counts of each set come from
        // the host's per-set counts (checked against int32 per set in batch_check), not from the whole concatenation
        int32_t rc = ensure_seq_counts(h, launches);
        if (rc) return rc;
        CUDA_TRY(b->pvals.reserve((size_t)b->n_seqs * m));
        for (int32_t s = 0; s < b->n_sets; ++s) {
            const int N = b->seq_off[s + 1] - b->seq_off[s], span = N * m;
            pvals_kernel<<<(span + 255) / 256, 256, 0, h->stream>>>(span, p->pseudocount, ppm_den(N, p), b->pvals.p + (size_t)m * b->seq_off[s]);
            CUDA_TRY(cudaGetLastError());
            int32_t g[4];
            for (int x = 0; x < 4; ++x) g[x] = (int32_t)b->gcnt[4 * (size_t)s + x];
            b->fast[s] = drift_fast_path_ok(g, batch_gap_total(b, p, s), b->max_len[s], N, p);
        }
        *launches += b->n_sets;
    }
    if (h->opt_exact_scans) b->fast.assign((size_t)b->n_sets, 0);
    b->tab_bgmode = p->background;
    b->tab_pc = p->pseudocount;
    b->tab_alen = p->alphabet_size;
    b->tab_k = p->k;
    b->tab_m = m;
    b->tab_bgwin = bg_win ? 1 : 0;
    b->tab_bg = bg;
    b->tab_valid = true;
    return GIBBS_OK;
}

// the result buffers of a run of R restarts per set, the statistics cleared
int32_t batch_results(gibbs_batch *b, int32_t R) {
    gibbs_handle *h = b->h;
    const size_t cells = (size_t)R * b->n_seqs;
    CUDA_TRY(h->sites.reserve(cells));
    CUDA_TRY(h->hv.reserve(cells));
    CUDA_TRY(h->scores.reserve(cells));
    CUDA_TRY(h->sums.reserve((size_t)b->n_sets * R));
    CUDA_TRY(h->stats.reserve(ST_NSLOTS));
    CUDA_TRY(cudaMemsetAsync(h->stats.p, 0, ST_NSLOTS * sizeof(unsigned long long), h->stream));
    return GIBBS_OK;
}

// the ChainArgs of set s: its rows and tables (m = motifAmount of the tables), its slices of the results
ChainArgs batch_set_args(const gibbs_batch *b, const gibbs_params *p, int32_t s, int32_t R, int m) {
    const gibbs_handle *h = b->h;
    const int32_t o = b->seq_off[s];
    const bool drift = p->background == GIBBS_BG_DATA;
    ChainArgs a;
    memset(&a, 0, sizeof a);
    a.s = batch_seqs(b, s);
    a.k = p->k;
    a.sampler = GIBBS_SITE_SAMPLER;
    a.n_chains = R;
    a.sites = h->sites.p + (size_t)R * o;
    a.hv = h->hv.p + (size_t)R * o;
    a.scores = h->scores.p + (size_t)R * o;
    a.sums = h->sums.p + (size_t)R * s;
    a.fast_ok = b->fast[s];
    if (drift) {
        a.pvals = b->pvals.p + (size_t)m * o;
        a.basecnt = h->basecnt.p + 4 * (size_t)o;
        a.maskcnt = b->n_masked[s] > 0 ? h->maskcnt.p + o : nullptr;
        a.ss = h->ss_valid ? h->ss.p + (size_t)o * (size_t)(h->max_len + 2) * 4 : nullptr;
        a.ss_stride = h->max_len + 2;
        for (int x = 0; x < 4; ++x) a.gcnt[x] = (int32_t)b->gcnt[4 * (size_t)s + x];
        a.gap_total = batch_gap_total(b, p, s);
        a.alpha_pc = (double)p->alphabet_size * p->pseudocount; // fs:117
        a.pc = p->pseudocount;
        a.drift_fast_ok = b->fast[s];
    } else {
        a.wtab = b->wtab.p + 4 * (size_t)m * o;
        memcpy(a.bg, b->tab_bg.data() + 4 * (size_t)s, sizeof a.bg);
    }
    return a;
}

// Launch groups: (masked symbols) x (4 warps per chain for sets of >= 4 sequences, else 1), then with all_sets one more
// group of every set (motifAmount = 2: one warp per restart). ids[g] = the sets of group g, at[g] = its offset in groups.
int32_t batch_groups(gibbs_batch *b, int32_t R, bool all_sets, std::vector<int32_t> *ids, size_t *at) {
    for (int32_t s = 0; s < b->n_sets; ++s) ids[(b->n_masked[s] > 0 ? 2 : 0) + (batch_team(b, s) == 4 ? 0 : 1)].push_back(s);
    if (all_sets)
        for (int32_t s = 0; s < b->n_sets; ++s) ids[BATCH_GROUPS].push_back(s);
    std::vector<int32_t> groups;
    for (int g = 0; g < BATCH_GROUPS + (all_sets ? 1 : 0); ++g) {
        at[g] = groups.size();
        groups.insert(groups.end(), ids[g].begin(), ids[g].end());
        for (size_t i = 0; i <= ids[g].size(); ++i) groups.push_back((int32_t)(i * (size_t)R));
    }
    if (groups != b->groups_host) {
        CUDA_TRY(b->d_groups.reserve(groups.size()));
        CUDA_TRY(cudaMemcpyAsync(b->d_groups.p, groups.data(), groups.size() * sizeof(int32_t), cudaMemcpyHostToDevice, b->h->stream));
        b->groups_host.swap(groups);
    }
    return GIBBS_OK;
}

// every group's random starts (chain_batch_kernel<.., INIT_ONLY>) or sweeps of a SiteSampler run
int32_t batch_launch_chains(gibbs_batch *b, const ChainArgs &run, bool drift, bool init, const std::vector<int32_t> *ids,
                            const size_t *at, int R, int *launches) {
    gibbs_handle *h = b->h;
    const long long per_sm = ((long long)b->n_sets * R + h->sm_count - 1) / h->sm_count;
    for (int g = 0; g < BATCH_GROUPS; ++g) {
        const int n = (int)ids[g].size();
        if (n == 0) continue;
        const bool masked = g >= 2;
        const int team = (g & 1) ? 1 : 4;
        if (!h->run_team) h->run_team = team;
        BatchTable bt;
        bt.sets = b->d_args.p;
        bt.set_ids = b->d_groups.p + at[g];
        bt.chain_off = b->d_groups.p + at[g] + n;
        bt.n = n;
        ChainArgs r = run;
        r.min_width = per_sm <= 1 ? team : 1; // (as plan_stages: never narrow once a chain has an SM to itself)
        BatchLaunch f;
        const int32_t rc = find_unit(BATCH_UNITS, "batch", team, masked, drift, init, &f);
        if (rc) return rc;
        CUDA_TRY(f(r, bt, n * R, team_smem_bytes(h->row_words, team), h->stream));
        ++*launches;
    }
    return GIBBS_OK;
}

// the argument checks of gibbs_batch_create that need no device (pointers and set_offsets)
int32_t batch_check_layout(const uint8_t *seqs, const int64_t *offsets, const int32_t *set_offsets, int32_t n_sets) {
    if (!seqs || !offsets || !set_offsets) return fail(GIBBS_ERR_ARG, "null sequence buffer or set offsets (ArgumentNullException)");
    if (n_sets < 1) return fail(GIBBS_ERR_ARG, "n_sets must be >= 1");
    if (set_offsets[0] != 0) return fail(GIBBS_ERR_ARG, "set_offsets[0] must be 0 (it is %d)", set_offsets[0]);
    for (int32_t s = 0; s < n_sets; ++s)
        if (set_offsets[s + 1] <= set_offsets[s])
            return fail(GIBBS_ERR_ARG, "set %d is empty or set_offsets decrease (%d .. %d)", s, set_offsets[s], set_offsets[s + 1]);
    return GIBBS_OK;
}

// gibbs_batch_create after batch_check_layout; the sets are sets set_base .. of set_total in the caller's numbering
int32_t batch_create(const uint8_t *seqs, const int64_t *offsets, const int32_t *set_offsets, int32_t n_sets, int32_t device,
                     int32_t set_base, int32_t set_total, gibbs_batch **out) {
    const int32_t n_seqs = set_offsets[n_sets];
    gibbs_batch *b = new (std::nothrow) gibbs_batch();
    if (!b) return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    try {
        b->seq_off.assign(set_offsets, set_offsets + n_sets + 1);
        b->min_len.assign((size_t)n_sets, INT32_MAX);
        b->max_len.assign((size_t)n_sets, 0);
        b->n_masked.assign((size_t)n_sets, 0);
        b->n_gap.assign((size_t)n_sets, 0);
        b->gcnt.assign((size_t)n_sets * 4, 0);
    } catch (...) {
        delete b;
        return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    }
    b->n_sets = n_sets;
    b->n_seqs = n_seqs;
    b->set_base = set_base;
    b->set_total = set_total;
    // per-set symbol classes; a failure names the set and the sequence (gibbs_create would only name the symbol)
    for (int32_t s = 0; s < n_sets; ++s) {
        for (int32_t i = set_offsets[s]; i < set_offsets[s + 1]; ++i) {
            const int64_t l = offsets[i + 1] - offsets[i];
            if (l < 0) {
                delete b;
                return fail(GIBBS_ERR_ARG, "set %d, sequence %d: offsets must be non-decreasing", set_base + s, i - set_offsets[s]);
            }
            if (l > GIBBS_MAX_LEN) {
                delete b;
                return fail(GIBBS_ERR_ARG, "set %d, sequence %d: longer than %d", set_base + s, i - set_offsets[s], GIBBS_MAX_LEN);
            }
            b->min_len[s] = std::min(b->min_len[s], (int32_t)l);
            b->max_len[s] = std::max(b->max_len[s], (int32_t)l);
            for (int64_t j = offsets[i]; j < offsets[i + 1]; ++j) {
                const uint8_t c = seqs[j];
                if (c == 'A') ++b->gcnt[4 * (size_t)s];
                else if (c == 'C') ++b->gcnt[4 * (size_t)s + 1];
                else if (c == 'G') ++b->gcnt[4 * (size_t)s + 2];
                else if (c == 'T') ++b->gcnt[4 * (size_t)s + 3];
                else if (c >= 42 && c <= 90) {
                    ++b->n_masked[s];
                    if (c == '-') ++b->n_gap[s];
                } else {
                    delete b;
                    return fail(GIBBS_ERR_SYMBOL, "set %d, sequence %d: symbol '%c' (0x%02x) is outside '*'..'Z', the range of the "
                                                  "49-slot tables (IndexOutOfRangeException, fs:17-20)",
                                set_base + s, i - set_offsets[s], c >= 32 && c < 127 ? (char)c : '?', c);
                }
            }
        }
    }
    int32_t rc = gibbs_create(seqs, offsets, n_seqs, device, &b->h);
    if (!rc) {
        gibbs_handle *h = b->h;
        cudaError_t e = b->d_seq_off.reserve((size_t)n_sets + 1);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(b->d_seq_off.p, b->seq_off.data(), b->seq_off.size() * sizeof(int32_t), cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) rc = fail(GIBBS_ERR_CUDA, "batch upload: %s", cudaGetErrorString(e));
    }
    if (rc) {
        gibbs_batch_destroy(b);
        return rc;
    }
    *out = b;
    return GIBBS_OK;
}

} // namespace

int32_t gibbs_batch_create(const uint8_t *seqs, const int64_t *offsets, const int32_t *set_offsets, int32_t n_sets, int32_t device,
                           gibbs_batch **out) {
    if (!out) return fail(GIBBS_ERR_ARG, "null out pointer");
    *out = nullptr;
    const int32_t rc = batch_check_layout(seqs, offsets, set_offsets, n_sets);
    if (rc) return rc;
    return batch_create(seqs, offsets, set_offsets, n_sets, device, 0, n_sets, out);
}

int32_t gibbs_batch_destroy(gibbs_batch *b) {
    if (!b) return GIBBS_OK;
    gibbs_handle *h = b->h;
    if (h) {
        cudaSetDevice(h->device);
        cudaStreamSynchronize(h->stream);
    }
    delete b; // the batch's device buffers, on the handle's device
    gibbs_destroy(h);
    return GIBBS_OK;
}

int32_t gibbs_batch_run_device(gibbs_batch *b, const gibbs_params *p, const double *bg_per_set, int32_t restarts_per_set,
                               int64_t chain_id_base, uint64_t seed) {
    int32_t rc = batch_check(b, p, bg_per_set, restarts_per_set, false);
    if (rc) return rc;
    gibbs_handle *h = b->h;
    rc = set_device(h);
    if (rc) return rc;
    h->run_done = false;
    const int32_t R = restarts_per_set, S = b->n_sets;
    const bool drift = p->background == GIBBS_BG_DATA;
    int launches = 0;
    rc = batch_tables(b, p, bg_per_set, 1, false, &launches);
    if (rc) return rc;
    rc = batch_results(b, R);
    if (rc) return rc;

    // run-wide arguments (chain_batch_kernel copies them over the set's own)
    ChainArgs run{};
    run.k = p->k;
    run.max_sweeps = p->max_sweeps > 0 ? p->max_sweeps : 1000000;
    run.sampler = GIBBS_SITE_SAMPLER;
    run.phase_mask = GIBBS_PHASE_GREEDY | (p->phase_shifts ? (GIBBS_PHASE_LEFT | GIBBS_PHASE_RIGHT) : 0);
    run.rng_mode = GIBBS_RNG_PHILOX;
    run.seed = seed;
    run.chain_id_base = chain_id_base;
    run.stats = h->stats.p;

    std::vector<ChainArgs> args((size_t)S);
    int fast_all = 1;
    for (int32_t s = 0; s < S; ++s) {
        args[s] = batch_set_args(b, p, s, R, 1);
        fast_all &= b->fast[s];
    }
    std::vector<int32_t> ids[BATCH_GROUPS];
    size_t g_at[BATCH_GROUPS];
    rc = batch_groups(b, R, false, ids, g_at);
    if (rc) return rc;
    rc = upload_if_changed(args, b->args_host, b->d_args, h->stream);
    if (rc) return rc;
    h->run_team = 0;
    CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
    for (int init = 1; init >= 0; --init) { // every group's random starts, then every group's sweeps
        rc = batch_launch_chains(b, run, drift, init != 0, ids, g_at, R, &launches);
        if (rc) return rc;
    }
    CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
    h->run_chains = R;
    h->run_k = p->k;
    h->run_fast = fast_all;
    h->run_launches = launches;
    h->run_init_path = GIBBS_INIT_CHAIN;
    h->run_sampler = GIBBS_SITE_SAMPLER;
    h->run_m = 1;
    h->best_valid = false;
    h->run_done = true;
    return GIBBS_OK;
}

int32_t gibbs_batch_run_motif_device(gibbs_batch *b, const gibbs_params *p, const double *bg_per_set, int32_t restarts_per_set,
                                     int64_t chain_id_base, uint64_t seed) {
    int32_t rc = batch_check(b, p, bg_per_set, restarts_per_set, true);
    if (rc) return rc;
    gibbs_handle *h = b->h;
    rc = set_device(h);
    if (rc) return rc;
    h->run_done = false;
    const int32_t R = restarts_per_set, S = b->n_sets, M = p->motif_amount == 2 ? 2 : 1;
    const bool drift = p->background == GIBBS_BG_DATA;
    int launches = 0;
    rc = batch_tables(b, p, bg_per_set, M, !drift, &launches);
    if (rc) return rc;
    rc = batch_results(b, R);
    if (rc) return rc;

    // scratch lists: set s holds R x T_s lists of its own window stride W_s (a 100 kb set does not widen the others')
    std::vector<size_t> scr((size_t)S + 1, 0);
    std::vector<int32_t> wstride((size_t)S);
    for (int32_t s = 0; s < S; ++s) {
        int W = b->max_len[s] - p->k + 1;
        if (drift && b->n_masked[s] > 0 && W < 64) W = 64; // the candidate scratch doubles as a 49-slot symbol-count table
        wstride[s] = W;
        scr[s + 1] = scr[s] + (size_t)R * (M == 2 ? 1 : batch_team(b, s)) * W;
    }
    const size_t cells = (size_t)R * b->n_seqs;
    CUDA_TRY(h->cand_l.reserve(scr[S]));
    CUDA_TRY(h->cand_w.reserve(scr[S]));
    if (drift) CUDA_TRY(h->gbuf.reserve(scr[S]));
    if (M == 2) {
        CUDA_TRY(h->sc2.reserve(scr[S]));
        CUDA_TRY(h->pos2.reserve(cells * 2));
    }
    CUDA_TRY(h->err_flag.reserve((size_t)S));
    CUDA_TRY(cudaMemsetAsync(h->err_flag.p, 0, (size_t)S * sizeof(int32_t), h->stream));

    // per-set arguments: the ChainArgs of the random starts and, around them, the MotifSampler's own
    std::vector<ChainArgs> args((size_t)S);
    std::vector<Motif2Args> margs((size_t)S);
    int fast_all = 1;
    for (int32_t s = 0; s < S; ++s) {
        const int32_t o = b->seq_off[s];
        ChainArgs &a = args[s];
        a = batch_set_args(b, p, s, R, M);
        a.sampler = GIBBS_MOTIF_SAMPLER;
        a.cutoff = p->cutoff;
        if (drift) a.fast_ok = 0; // (as gibbs_run_device: the data-derived background's range check is drift_fast_ok)
        fast_all &= b->fast[s];
        Motif2Args &q = margs[s];
        memset(&q, 0, sizeof q);
        MotifArgs &m = q.m;
        m.c = a;
        if (!drift) {
            m.bg.g = b->bg_g.p + b->g_off[s];
            m.bg.gsum = b->bg_sum.p + o;
            m.bg.gmax = b->bg_max.p + o;
            m.bg.gmax_i = b->bg_max_i.p + o;
        }
        m.bg.wstride = wstride[s];
        m.cand_l = h->cand_l.p + scr[s];
        m.cand_w = h->cand_w.p + scr[s];
        m.error = h->err_flag.p + s;
        m.data_bg = drift ? 1 : 0;
        m.greedy_fast_ok = b->fast[s];
        if (drift) {
            m.pvals = a.pvals;
            m.basecnt = a.basecnt;
            memcpy(m.gcnt, a.gcnt, sizeof m.gcnt);
            m.alpha_pc = a.alpha_pc;
            m.pc = a.pc;
            m.gbuf = h->gbuf.p + scr[s];
        }
        m.roulette_scan_ok = h->opt_exact_scans ? 0 : 1;
        m.ascii = h->ascii.p;
        m.off = h->off.p + o;
        if (M == 2) {
            q.pos2 = h->pos2.p + 2 * (size_t)R * o;
            q.sc = h->sc2.p + scr[s];
        }
    }
    std::vector<int32_t> ids[BATCH_GROUPS + 1];
    size_t g_at[BATCH_GROUPS + 1];
    rc = batch_groups(b, R, M == 2, ids, g_at);
    if (rc) return rc;
    rc = upload_if_changed(args, b->args_host, b->d_args, h->stream);
    if (rc) return rc;
    rc = upload_if_changed(margs, b->margs_host, b->d_margs, h->stream);
    if (rc) return rc;

    // run-wide arguments: the random starts are the SiteSampler's (fs:876, fs:993), then the stochastic and greedy sweeps
    ChainArgs run{};
    run.k = p->k;
    run.max_sweeps = p->max_sweeps > 0 ? p->max_sweeps : 1000000;
    run.sampler = GIBBS_MOTIF_SAMPLER;
    run.phase_mask = GIBBS_PHASE_INIT | GIBBS_PHASE_STOCHASTIC | GIBBS_PHASE_MOTIF_GREEDY;
    run.rng_mode = GIBBS_RNG_PHILOX;
    run.seed = seed;
    run.chain_id_base = chain_id_base;
    run.stats = h->stats.p;
    MotifArgs mrun{};
    mrun.c = run;
    mrun.c.phase_mask = GIBBS_PHASE_STOCHASTIC | GIBBS_PHASE_MOTIF_GREEDY;
    mrun.c.cutoff = p->cutoff;
    mrun.init_done = 1;
    h->run_team = 0;
    CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
    rc = batch_launch_chains(b, run, drift, true, ids, g_at, R, &launches);
    if (rc) return rc;
    if (M == 2) {
        const int n = (int)ids[BATCH_GROUPS].size();
        const MotifBatchTable bt{b->d_margs.p, b->d_groups.p + g_at[BATCH_GROUPS], b->d_groups.p + g_at[BATCH_GROUPS] + n, n};
        CUDA_TRY(launch_motif2_batch(mrun, bt, n * R, team_smem_bytes(h->row_words, 1), h->stream));
        ++launches;
        h->run_team = 1;
    } else {
        h->run_team = 0;
        for (int g = 0; g < BATCH_GROUPS; ++g) {
            const int n = (int)ids[g].size();
            if (n == 0) continue;
            const bool masked = g >= 2;
            const int team = (g & 1) ? 1 : 4;
            if (!h->run_team) h->run_team = team;
            const MotifBatchTable bt{b->d_margs.p, b->d_groups.p + g_at[g], b->d_groups.p + g_at[g] + n, n};
            MotifBatchLaunch f;
            rc = find_unit(MOTIF_BATCH_UNITS, "MotifSampler batch", team, masked, false, false, &f);
            if (rc) return rc;
            CUDA_TRY(f(mrun, bt, n * R, team_smem_bytes(h->row_words, team), h->stream));
            ++launches;
        }
    }
    CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
    h->run_chains = R;
    h->run_k = p->k;
    h->run_fast = fast_all;
    h->run_launches = launches;
    h->run_init_path = GIBBS_INIT_CHAIN;
    h->run_sampler = GIBBS_MOTIF_SAMPLER;
    h->run_m = M;
    h->best_valid = false;
    h->run_done = true;
    return GIBBS_OK;
}

static void batch_stats(const gibbs_handle *h, const unsigned long long *st, int extra_launches, gibbs_run_stats *out) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) cudaGetLastError();
    fill_stats(out, st, h->run_launches + extra_launches, h->run_fast, h->run_team, h->run_init_path, ms);
}

int32_t gibbs_batch_fetch(gibbs_batch *b, int32_t *sites_out, double *scores_out, double *sums_out, gibbs_run_stats *stats_out) {
    if (!b) return fail(GIBBS_ERR_ARG, "null batch");
    gibbs_handle *h = b->h;
    if (!h->run_done) return fail(GIBBS_ERR_ARG, "gibbs_batch_fetch without a preceding gibbs_batch_run_device");
    int32_t rc = set_device(h);
    if (rc) return rc;
    const size_t cells = (size_t)h->run_chains * b->n_seqs;
    if (sites_out) CUDA_TRY(cudaMemcpyAsync(sites_out, h->sites.p, cells * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (scores_out) CUDA_TRY(cudaMemcpyAsync(scores_out, h->scores.p, cells * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (sums_out)
        CUDA_TRY(cudaMemcpyAsync(sums_out, h->sums.p, (size_t)h->run_chains * b->n_sets * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    unsigned long long st[ST_NSLOTS];
    CUDA_TRY(cudaMemcpyAsync(st, h->stats.p, sizeof st, cudaMemcpyDeviceToHost, h->stream));
    rc = sync_roulette(h, b->n_sets, b->set_base);
    if (rc) return rc;
    if (stats_out) batch_stats(h, st, 0, stats_out);
    return GIBBS_OK;
}

int32_t gibbs_batch_fetch_best(gibbs_batch *b, int32_t repetitions, int32_t *sites_out, double *scores_out, int32_t *n_out,
                               double *sum_out, int32_t *restart_out, int32_t *counts_out, gibbs_run_stats *stats_out) {
    if (!b) return fail(GIBBS_ERR_ARG, "null batch");
    gibbs_handle *h = b->h;
    if (!h->run_done) return fail(GIBBS_ERR_ARG, "gibbs_batch_fetch_best without a preceding gibbs_batch_run_device");
    if (repetitions < 0) repetitions = 0;
    int32_t rc = set_device(h);
    if (rc) return rc;
    const int32_t S = b->n_sets, k = h->run_k;
    auto select = [&](const int32_t *sites, int m, int motif, int32_t *best_out, double *win_sums) -> int32_t {
        restart_select_batch_kernel<<<S, 32, 0, h->stream>>>(h->sums.p, sites, h->scores.p, b->d_seq_off.p, h->run_chains, repetitions, m,
                                                            motif, best_out, h->win_sites.p, h->win_scores.p, win_sums);
        CUDA_TRY(cudaGetLastError());
        return GIBBS_OK;
    };
    auto counts = [&](const int32_t *sites, int32_t *out) {
        return with_kp(k, [&](auto kp) -> int32_t {
            all_counts_batch_kernel<kp()><<<S, 32, 0, h->stream>>>(b->d_args.p, b->d_seq_off.p, sites, k, out);
            CUDA_TRY(cudaGetLastError());
            return GIBBS_OK;
        });
    };
    unsigned long long st[ST_NSLOTS];
    int extra_launches = 0;
    rc = fetch_winners(h, S, b->seq_off.data(), b->set_base, select, counts, sites_out, scores_out, n_out, sum_out, restart_out,
                       counts_out, st, &extra_launches);
    if (rc) return rc;
    if (stats_out) batch_stats(h, st, extra_launches, stats_out);
    return GIBBS_OK;
}

int32_t gibbs_batch_fetch_positions(gibbs_batch *b, int32_t m, int32_t *positions_out) {
    if (!b || !positions_out) return fail(GIBBS_ERR_ARG, "null argument");
    return fetch_positions(b->h, m, positions_out, "gibbs_batch_fetch_positions without a preceding run");
}

int32_t gibbs_batch_fetch_best_positions(gibbs_batch *b, int32_t m, int32_t *positions_out) {
    if (!b || !positions_out) return fail(GIBBS_ERR_ARG, "null argument");
    return fetch_best_positions(b->h, m, positions_out, "gibbs_batch_fetch_best_positions without a preceding gibbs_batch_fetch_best");
}

/* ---- many sequence sets over several devices ----------------------------------------------------------------------- */
// The sets are split once, at create time, into contiguous blocks, one per device slot; each slot holds an ordinary
// gibbs_batch over its block (no set is replicated). Its set_base / set_total make its checks and messages those of one
// batch over all the sets, and set s gives bit for bit what it gives in any batch, so the results are the one-device
// batch's whatever the split.
struct gibbs_multi_batch {
    std::vector<gibbs_batch *> slot;   // nullptr: an empty slot (fewer sets than slots)
    std::vector<int32_t> first, count; // slot i holds sets first[i] .. first[i] + count[i] - 1
    std::vector<int32_t> set_off;      // [n_sets + 1] the caller's set_offsets
    int32_t run_R = 0, run_k = 0;
    bool run_done = false, best_valid = false;
};

namespace {

// Contiguous blocks of sets, one per slot, whose largest cost is the least possible. The cost of a set is the sum of its
// sequence lengths: up to k - 1 per sequence, the windows one sweep of one restart scores (k, the restart count and the
// sampler are not known at create time). The least feasible bound is found by binary search over a greedy block count;
// the blocks are then filled from the left up to it, keeping one set for each later slot while there are enough, so a
// slot is left empty only when there are fewer sets than slots.
void partition_sets(const std::vector<int64_t> &cost, int32_t slots, std::vector<int32_t> &first, std::vector<int32_t> &count) {
    const int32_t S = (int32_t)cost.size();
    int64_t lo = 0, hi = 0;
    for (const int64_t c : cost) {
        lo = std::max(lo, c);
        hi += c;
    }
    while (lo < hi) { // least bound whose greedy blocks number at most `slots`
        const int64_t mid = lo + (hi - lo) / 2;
        int32_t blocks = 1;
        int64_t sum = 0;
        for (const int64_t c : cost) {
            if (sum + c > mid) {
                ++blocks;
                sum = 0;
            }
            sum += c;
        }
        if (blocks <= slots) hi = mid;
        else lo = mid + 1;
    }
    first.assign((size_t)slots, S);
    count.assign((size_t)slots, 0);
    int32_t next = 0;
    for (int32_t i = 0; i < slots && next < S; ++i) {
        first[i] = next;
        int64_t sum = 0;
        do {
            sum += cost[next++];
        } while (next < S && sum + cost[next] <= lo && S - next > slots - i - 1);
        count[i] = next - first[i];
    }
}

// the sum of the slots' statistics: counters and launches added, kernel_ms the slowest slot (the devices run concurrently),
// the other fields those of the first slot
void add_slot_stats(gibbs_run_stats &total, const gibbs_run_stats &st, bool first_slot) {
    if (first_slot) total = st;
    else {
        total.site_updates += st.site_updates;
        total.window_scores += st.window_scores;
        total.sweeps += st.sweeps;
        total.exact_rescans += st.exact_rescans;
        total.capped_chains += st.capped_chains;
        total.speculative_discards += st.speculative_discards;
        total.kernel_launches += st.kernel_launches;
        total.kernel_ms = std::max(total.kernel_ms, st.kernel_ms);
    }
}

// checks the run on every slot first -- in set order, so a failure is the one a batch over all the sets reports -- then
// queues each slot's run on its device without waiting for any of them
int32_t multi_batch_run(gibbs_multi_batch *mb, const gibbs_params *p, const double *bg_per_set, int32_t R, int64_t chain_id_base,
                        uint64_t seed, bool motif) {
    if (!mb) return fail(GIBBS_ERR_ARG, "null multi-device batch");
    mb->run_done = mb->best_valid = false;
    for (size_t i = 0; i < mb->slot.size(); ++i) {
        if (!mb->slot[i]) continue;
        const int32_t rc = batch_check(mb->slot[i], p, bg_per_set ? bg_per_set + 4 * (size_t)mb->first[i] : nullptr, R, motif);
        if (rc) return rc;
    }
    for (size_t i = 0; i < mb->slot.size(); ++i) {
        if (!mb->slot[i]) continue;
        const double *bg = bg_per_set ? bg_per_set + 4 * (size_t)mb->first[i] : nullptr;
        const int32_t rc = motif ? gibbs_batch_run_motif_device(mb->slot[i], p, bg, R, chain_id_base, seed)
                                 : gibbs_batch_run_device(mb->slot[i], p, bg, R, chain_id_base, seed);
        if (rc) return rc;
    }
    mb->run_R = R;
    mb->run_k = p->k;
    mb->run_done = true;
    return GIBBS_OK;
}

} // namespace

int32_t gibbs_multi_batch_create(const uint8_t *seqs, const int64_t *offsets, const int32_t *set_offsets, int32_t n_sets,
                                 const int32_t *devices, int32_t n_devices, gibbs_multi_batch **out) {
    if (!out) return fail(GIBBS_ERR_ARG, "null out pointer");
    *out = nullptr;
    int32_t rc = batch_check_layout(seqs, offsets, set_offsets, n_sets);
    if (rc) return rc;
    if (n_devices < 0) return fail(GIBBS_ERR_ARG, "n_devices = %d must be >= 0", n_devices);
    const int32_t visible = gibbs_device_count();
    if (visible < 1) return fail(GIBBS_ERR_CUDA, "no CUDA device available; libgibbs_b200 has no CPU fallback");
    if (n_devices == 0) n_devices = visible; // 0 = every visible device
    // (an explicit device list may name a device twice: two slots then share it)
    if (!devices && n_devices > visible) return fail(GIBBS_ERR_ARG, "n_devices = %d, %d visible", n_devices, visible);
    gibbs_multi_batch *mb = new (std::nothrow) gibbs_multi_batch();
    if (!mb) return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    std::vector<int32_t> so;
    try {
        std::vector<int64_t> cost((size_t)n_sets, 0);
        for (int32_t s = 0; s < n_sets; ++s)
            for (int32_t i = set_offsets[s]; i < set_offsets[s + 1]; ++i)
                cost[s] += std::max<int64_t>(offsets[i + 1] - offsets[i], 0); // (bad offsets are reported by the slot's batch)
        partition_sets(cost, n_devices, mb->first, mb->count);
        mb->set_off.assign(set_offsets, set_offsets + n_sets + 1);
        mb->slot.assign((size_t)n_devices, nullptr);
    } catch (...) {
        delete mb;
        return fail(GIBBS_ERR_NOMEM, "host allocation failed");
    }
    for (int32_t i = 0; i < n_devices; ++i) {
        const int32_t f = mb->first[i], c = mb->count[i];
        if (c == 0) continue;
        try {
            so.resize((size_t)c + 1);
        } catch (...) {
            gibbs_multi_batch_destroy(mb);
            return fail(GIBBS_ERR_NOMEM, "host allocation failed");
        }
        for (int32_t s = 0; s <= c; ++s) so[s] = set_offsets[f + s] - set_offsets[f];
        rc = batch_create(seqs, offsets + set_offsets[f], so.data(), c, devices ? devices[i] : i, f, n_sets, &mb->slot[i]);
        if (rc) {
            gibbs_multi_batch_destroy(mb);
            return rc;
        }
    }
    *out = mb;
    return GIBBS_OK;
}

int32_t gibbs_multi_batch_destroy(gibbs_multi_batch *mb) {
    if (!mb) return GIBBS_OK;
    for (gibbs_batch *b : mb->slot) gibbs_batch_destroy(b);
    delete mb;
    return GIBBS_OK;
}

int32_t gibbs_multi_batch_num_devices(const gibbs_multi_batch *mb) { return mb ? (int32_t)mb->slot.size() : 0; }

int32_t gibbs_multi_batch_slot_sets(const gibbs_multi_batch *mb, int32_t slot, int32_t *first_set_out, int32_t *n_sets_out) {
    if (!mb || !first_set_out || !n_sets_out) return fail(GIBBS_ERR_ARG, "null argument");
    if (slot < 0 || slot >= (int32_t)mb->slot.size()) return fail(GIBBS_ERR_ARG, "slot %d outside 0..%d", slot, (int)mb->slot.size() - 1);
    *first_set_out = mb->first[slot];
    *n_sets_out = mb->count[slot];
    return GIBBS_OK;
}

int32_t gibbs_multi_batch_run_device(gibbs_multi_batch *mb, const gibbs_params *p, const double *bg_per_set, int32_t restarts_per_set,
                                     int64_t chain_id_base, uint64_t seed) {
    return multi_batch_run(mb, p, bg_per_set, restarts_per_set, chain_id_base, seed, false);
}

int32_t gibbs_multi_batch_run_motif_device(gibbs_multi_batch *mb, const gibbs_params *p, const double *bg_per_set,
                                           int32_t restarts_per_set, int64_t chain_id_base, uint64_t seed) {
    return multi_batch_run(mb, p, bg_per_set, restarts_per_set, chain_id_base, seed, true);
}

int32_t gibbs_multi_batch_fetch(gibbs_multi_batch *mb, int32_t *sites_out, double *scores_out, double *sums_out,
                                gibbs_run_stats *stats_out) {
    if (!mb) return fail(GIBBS_ERR_ARG, "null multi-device batch");
    if (!mb->run_done) return fail(GIBBS_ERR_ARG, "gibbs_multi_batch_fetch without a preceding run");
    gibbs_run_stats total{};
    bool first_slot = true;
    for (size_t i = 0; i < mb->slot.size(); ++i) {
        if (!mb->slot[i]) continue;
        const size_t rows = (size_t)mb->run_R * mb->set_off[mb->first[i]], sums = (size_t)mb->run_R * mb->first[i];
        gibbs_run_stats st{};
        const int32_t rc = gibbs_batch_fetch(mb->slot[i], sites_out ? sites_out + rows : nullptr, scores_out ? scores_out + rows : nullptr,
                                             sums_out ? sums_out + sums : nullptr, &st);
        if (rc) return rc;
        add_slot_stats(total, st, first_slot);
        first_slot = false;
    }
    if (stats_out) *stats_out = total;
    return GIBBS_OK;
}

int32_t gibbs_multi_batch_fetch_best(gibbs_multi_batch *mb, int32_t repetitions, int32_t *sites_out, double *scores_out, int32_t *n_out,
                                     double *sum_out, int32_t *restart_out, int32_t *counts_out, gibbs_run_stats *stats_out) {
    if (!mb) return fail(GIBBS_ERR_ARG, "null multi-device batch");
    if (!mb->run_done) return fail(GIBBS_ERR_ARG, "gibbs_multi_batch_fetch_best without a preceding run");
    mb->best_valid = false;
    gibbs_run_stats total{};
    bool first_slot = true;
    for (size_t i = 0; i < mb->slot.size(); ++i) { // the slots in set order: a roulette failure names the lowest failing set
        if (!mb->slot[i]) continue;
        const size_t f = (size_t)mb->first[i], o = (size_t)mb->set_off[f];
        gibbs_run_stats st{};
        const int32_t rc = gibbs_batch_fetch_best(mb->slot[i], repetitions, sites_out ? sites_out + o : nullptr, scores_out ? scores_out + o : nullptr,
                                                  n_out ? n_out + f : nullptr, sum_out ? sum_out + f : nullptr,
                                                  restart_out ? restart_out + f : nullptr,
                                                  counts_out ? counts_out + f * mb->run_k * 4 : nullptr, &st);
        if (rc) return rc;
        add_slot_stats(total, st, first_slot);
        first_slot = false;
    }
    mb->best_valid = true;
    if (stats_out) *stats_out = total;
    return GIBBS_OK;
}

int32_t gibbs_multi_batch_fetch_positions(gibbs_multi_batch *mb, int32_t m, int32_t *positions_out) {
    if (!mb || !positions_out) return fail(GIBBS_ERR_ARG, "null argument");
    if (!mb->run_done) return fail(GIBBS_ERR_ARG, "gibbs_multi_batch_fetch_positions without a preceding run");
    for (size_t i = 0; i < mb->slot.size(); ++i) {
        if (!mb->slot[i]) continue;
        const int32_t rc = gibbs_batch_fetch_positions(mb->slot[i], m, positions_out + (size_t)m * mb->run_R * mb->set_off[mb->first[i]]);
        if (rc) return rc;
    }
    return GIBBS_OK;
}

int32_t gibbs_multi_batch_fetch_best_positions(gibbs_multi_batch *mb, int32_t m, int32_t *positions_out) {
    if (!mb || !positions_out) return fail(GIBBS_ERR_ARG, "null argument");
    if (!mb->run_done || !mb->best_valid)
        return fail(GIBBS_ERR_ARG, "gibbs_multi_batch_fetch_best_positions without a preceding gibbs_multi_batch_fetch_best");
    for (size_t i = 0; i < mb->slot.size(); ++i) {
        if (!mb->slot[i]) continue;
        const int32_t rc = gibbs_batch_fetch_best_positions(mb->slot[i], m, positions_out + (size_t)m * mb->set_off[mb->first[i]]);
        if (rc) return rc;
    }
    return GIBBS_OK;
}

} // extern "C"
