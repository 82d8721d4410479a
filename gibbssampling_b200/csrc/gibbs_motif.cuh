// gibbssampling_b200/csrc/gibbs_motif.cuh -- MotifSampler, motifAmount = 1 (fs:709-1038): candidate list,
// roulette-wheel pick, the synchronous stochastic sweep and the greedy sweeps. A team of warps runs one chain
// (motif_kernel below); the stochastic sweep scores every window in float64 because the candidate list needs
// every window above the cut-off, not just the maximum.
//
// MotifIndex state per sequence: site (-1 = Positions []) and PWMS (log2 score of the site, or the raw
// background probability of a window when "no site" was picked, fs:774-777).
#pragma once
#include "gibbs_device.cuh"
#include "gibbs_kernels.cuh"
#include "gibbs_drift.cuh"

#ifndef GIBBS_MOTIF_NARROW_SWEEPS
#define GIBBS_MOTIF_NARROW_SWEEPS 1 // greedy sweeps whose speculative rounds may narrow after a discard (C2: 0 / 1 / 2 / 3 / all = 28.4 / 26.6 / 26.8 / 27.1 / 29.0 ms per step)
#endif
namespace gibbs {

enum MotifPhase { MPH_INIT = 0, MPH_STOCH = 1, MPH_GREEDY = 2, MPH_DONE = 3 };

// background-only window probabilities depend on the sequence and the fixed pcv only: computed once
struct BgTables {
    const double *g;       // [n][wstride] calculateSegmentScoreBy pcv window (fs:123-124, fs:776)
    const double *gsum;    // [n] sequential sum of g (the List.sum partial after the background entries, fs:748)
    const double *gmax;    // [n] first maximum of g ...
    const int32_t *gmax_i; // [n] ... and its window (List.sortByDescending is stable, fs:812)
    int32_t wstride;
};

struct MotifArgs {
    ChainArgs c;
    BgTables bg;           // fixed background: run constants
    double *cand_l;        // [chains][wstride] candidate PWMS scratch (ascending window order)
    int32_t *cand_w;       // [chains][wstride]
    int32_t *error;        // set to 1 when a roulette pick ran past the list (fs:753)
    // data-derived background (fs:885-970): one background per held-out sequence, built from the others'
    // bases outside their sites plus the whole held-out sequence (fs:896-905)
    int32_t data_bg;
    const double *pvals;   // [n] (c + pc) / ((N-1) + |A| pc)
    const int32_t *basecnt; // [n][4]
    int32_t gcnt[4];
    double alpha_pc, pc;
    double *gbuf;          // [chains][wstride] background window probabilities of the current held-out sequence
    int32_t greedy_fast_ok; // greedy sweeps may rank windows in fixed point (no float64 under/overflow possible, pc > 0)
    int32_t roulette_scan_ok; // stochastic sweep may locate the roulette bucket with a warp scan (0 = always walk)
    int32_t init_done;      // the random starts already ran (grid-wide kernel): sites + raw products in hv are the state
    // sets with symbols outside A,C,G,T, data-derived background: the uploaded symbols (see masked_background_window)
    const uint8_t *ascii;
    const int64_t *off;
};

// Background-only probability of a window that holds symbols outside the alphabet, data-derived background. The
// held-out sequence adds ALL its symbols to the count vector (fs:953) and createNormalizedPCVOfFCV normalises the
// alphabet slots only (fs:115-119): a symbol outside the alphabet keeps its raw count as its "probability", and
// calculateSegmentScoreBy multiplies it in like any other (fs:123-124). symc = the 49 symbol counts of the sequence.
static __device__ __noinline__ double masked_background_window(const uint8_t *seq, int w, int k, const double *q, const int32_t *symc) {
    double v = 1.0;
    for (int j = 0; j < k; ++j) {
        const int c = seq[w + j];
        const double f = c == 'A' ? q[0] : c == 'C' ? q[1] : c == 'G' ? q[2] : c == 'T' ? q[3] : (double)__ldcg(symc + (c - 42));
        v = __dmul_rn(v, f);
    }
    return v;
}

// one thread per sequence
static __global__ void bg_setup_kernel(DeviceSeqs s, int k, double q0, double q1, double q2, double q3, int wstride, double *g,
                                double *gsum, double *gmax, int32_t *gmax_i) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= s.n) return;
    const uint32_t *row = s.packed + (size_t)n * s.row_words;
    const uint32_t *mrow = (s.mask != nullptr && s.rowflag[n] != 0) ? s.mask + (size_t)n * s.row_words : nullptr;
    const int W = s.len[n] - k + 1;
    double sum = 0.0, best = 0.0;
    int best_i = 0;
    for (int w = 0; w < W; ++w) {
        double v = 1.0;
        for (int j = 0; j < k; ++j) {
            const int pos = w + j;
            const int b = (row[pos >> 4] >> ((pos & 15) * 2)) & 3;
            double q = b == 0 ? q0 : b == 1 ? q1 : b == 2 ? q2 : q3;
            if (mrow != nullptr && ((mrow[pos >> 4] >> ((pos & 15) * 2)) & 1u)) q = 0.0; // pcv of a symbol outside the alphabet (fs:115-119)
            v = __dmul_rn(v, q);
        }
        g[(size_t)n * wstride + w] = v;
        sum = __dadd_rn(sum, v);
        if (w == 0 || v > best) {
            best = v;
            best_i = w;
        }
    }
    gsum[n] = sum;
    gmax[n] = best;
    gmax_i[n] = best_i;
}

// calculateNormalizedSegmentScores (fs:759-784), motifAmount = 1, in two passes.
// Pass 1 (motif_gate): every window's float64 product; the windows above a cheap gate just below 2^cutOff are compacted
// (in window order) into cand_l (raw products) / cand_w, so that the logarithms -- ~150 instructions each, executed by the
// whole warp whenever one lane needs one -- are taken over a dense list instead of over all W windows. Returns their number.
// MASKED, masked_n >= 0: the sequence holds symbols outside A,C,G,T; a window over one scores 0 (PWM row 0, fs:283-287),
// log2 0 = -inf is never above the cut-off
template <int KP, bool MASKED = false>
__device__ __forceinline__ int motif_gate(const WarpTables &T, const uint32_t *row, int W, int k, double raw_gate, double *cand_l,
                                          int32_t *cand_w, int lane, const DeviceSeqs *sq = nullptr, int masked_n = -1) {
    int gated = 0;
    for (int w0 = 0; w0 < W; w0 += 32) {
        const int w = w0 + lane;
        double s = w < W ? exact_window<KP>(row, w, k, T.wcol) : 0.0;
        if (MASKED && masked_n >= 0 && w < W && mask_kmer(sq->mask, sq->row_words, masked_n, w, k) != 0) s = 0.0;
        const bool g = w < W && s > raw_gate; // (raw_gate >= 0: a masked window never passes)
        const unsigned m = __ballot_sync(FULL, g);
        if (g) {
            const int at = gated + __popc(m & ((1u << lane) - 1u));
            cand_l[at] = s;
            cand_w[at] = w;
        }
        gated += __popc(m);
    }
    __syncwarp();
    return gated;
}

// Pass 2 (motif_logs): the decision itself is made on the log (fs:735); the size-1 candidates, ascending position, each
// with log2(score) > cutOff, are compacted in place (a block writes only below what it has read) with their PWMS in
// cand_l. Returns their number and the first maximum by PWMS among them (best_l = -inf when there is none).
__device__ __forceinline__ int motif_logs(double cutoff, double *cand_l, int32_t *cand_w, int gated, int lane, double &best_l,
                                          int &best_w) {
    int count = 0;
    double bl = -INFINITY;
    int bw = INT32_MAX;
    for (int i0 = 0; i0 < gated; i0 += 32) {
        const int i = i0 + lane;
        double l = 0.0;
        int w = 0;
        bool is_c = false;
        if (i < gated) {
            l = log2_ref(cand_l[i]);
            w = cand_w[i];
            is_c = l > cutoff;
        }
        __syncwarp();
        const unsigned m = __ballot_sync(FULL, is_c);
        if (is_c) {
            const int at = count + __popc(m & ((1u << lane) - 1u));
            cand_l[at] = l;
            cand_w[at] = w;
            if (l > bl) { // ascending windows per lane: strict > keeps the first maximum
                bl = l;
                bw = w;
            }
        }
        count += __popc(m);
    }
    warp_argmax(bl, bw); // (largest PWMS, lowest window)
    best_l = bl;
    best_w = bw;
    __syncwarp();
    return count;
}

template <int KP, bool MASKED = false>
__device__ __forceinline__ int motif_candidates(const WarpTables &T, const uint32_t *row, int W, int k, double cutoff,
                                                double raw_gate, double *cand_l, int32_t *cand_w, int lane,
                                                double &best_l, int &best_w, const DeviceSeqs *sq = nullptr, int masked_n = -1) {
    const int gated = motif_gate<KP, MASKED>(T, row, W, k, raw_gate, cand_l, cand_w, lane, sq, masked_n);
    return motif_logs(cutoff, cand_l, cand_w, gated, lane, best_l, best_w);
}

// The roulette pick of the stochastic sweep without a float64 logarithm per candidate. log2 of a gated product to 1e-6:
// exponent + MUFU.LG2 of the float mantissa, added in double (exact: an integer below 2^11 plus a float in [0, 1]), so
// |error| < 4.5e-7 for any normal product at any magnitude -- MUFU.LG2's 2^-21.4 on [1, 2] plus 2^-24 / ln 2 for rounding
// the mantissa to float. (A float sum would round to half a float ulp of the result on top: 1.9e-6 above 32, 3.8e-6
// above 64, enough to put a window on the wrong side of the cut-off.) With those weights the candidates are decided
// (further than 1e-6 from the cut-off, else the exact path runs), their prefix sums locate the bucket of the pick, and
// the error of any prefix -- (items + 64) * 1e-6 -- is far below a bucket width (a candidate weighs more than the
// cut-off): when the pick clears both edges of its bucket by twice that bound the sequential float64 walk of
// fs:746-754 must stop in the same bucket, and only that item's PWMS is computed with the reference's logarithm.
// Needs cutOff >= 0 (no negative weights). false = undecided: the caller runs motif_logs + motif_roulette on the same list.
__device__ __forceinline__ double log2_coarse(double s) {
    const int hi = __double2hiint(s);
    const int e = ((hi >> 20) & 0x7ff) - 1023;
    const float m = (float)__hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(s)); // mantissa in [1, 2]
    return (double)e + (double)__log2f(m);
}
__device__ __forceinline__ bool motif_stoch_fast(double gsum, double cutoff, const double *cand_l, const int32_t *cand_w, int gated,
                                                 double pick, int lane, double &pwms_out, int &site_out) {
    constexpr double TOL = 1e-6;
    if (gated == 0 || !(cutoff >= 0.0) || !(gsum >= 0.0)) return false;
    const int B = (gated + 31) >> 5;
    const int i0 = min(gated, lane * B), i1 = min(gated, i0 + B);
    double part = 0.0;
    bool unsure = false;
    for (int i = i0; i < i1; ++i) {
        const double s = cand_l[i];
        const double l = log2_coarse(s);
        unsure |= !(s >= 0x1p-1000 && s <= 0x1p1000) || fabs(l - cutoff) <= TOL;
        if (l > cutoff) part += l;
    }
    if (__ballot_sync(FULL, unsure)) return false;
    double incl = part; // inclusive scan of the block sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    const double total = gsum + __shfl_sync(FULL, incl, 31);
    const double err = 2.0 * ((double)(gated + 64) * TOL + total * 0x1p-40);
    const double target = pick * total;
    if (!(target > gsum + err) || !(total < INFINITY)) return false; // background entries (1e-4 of the mass at most): exact path
    const unsigned holds = __ballot_sync(FULL, i0 < i1 && target <= gsum + incl);
    if (!holds) return false;
    const int src = __ffs(holds) - 1;
    int idx = -1;
    if (lane == src) {
        double acc = gsum + incl - part;
        for (int i = i0; i < i1; ++i) {
            const double l = log2_coarse(cand_l[i]);
            if (!(l > cutoff)) continue;
            const double nxt = acc + l;
            if (target <= nxt) {
                if (target > acc + err && target < nxt - err) idx = i;
                break;
            }
            acc = nxt;
        }
    }
    idx = __shfl_sync(FULL, idx, src);
    if (idx < 0) return false;
    pwms_out = log2_ref(cand_l[idx]);
    site_out = cand_w[idx];
    return true;
}

// rouletteWheelSelection (fs:746-754) over [W background entries] ++ [candidates]: exact sequential
// float64 semantics (sum from 0.0 in list order, weights PWMS/sum, inclusive bounds on both sides).
// Returns false when the pick ran past the list (the reference throws, fs:753).
static __device__ __noinline__ bool motif_roulette_exact(const double *g, double gsum, int W, const double *cand_l,
                                                  const int32_t *cand_w, int n_cand, double pick, int lane, double &pwms_out,
                                                  int &site_out) {
    double sum = gsum; // the background entries come first in the list; gsum was accumulated in that order
    for (int i = 0; i < n_cand; ++i) sum = __dadd_rn(sum, cand_l[i]);
    double acc = 0.0;
    const int total = W + n_cand;
    for (int i0 = 0; i0 < total; i0 += 32) {
        const int i = i0 + lane;
        double v = 0.0;
        if (i < total) v = (i < W) ? g[i] : cand_l[i - W];
        const double wgt = __ddiv_rn(v, sum); // divisions in parallel, accumulation in list order
        const int lim = min(32, total - i0);
        for (int j = 0; j < lim; ++j) {
            const double wj = __shfl_sync(FULL, wgt, j);
            const double hi = __dadd_rn(acc, wj);
            if (acc <= pick && pick <= hi) {
                const int idx = i0 + j;
                if (idx < W) {
                    pwms_out = g[idx];
                    site_out = -1;
                } else {
                    pwms_out = cand_l[idx - W];
                    site_out = cand_w[idx - W];
                }
                return true;
            }
            acc = hi;
        }
    }
    return false;
}

// ------------------------------------------------------------------------------------------------
// greedy sweeps (fs:788-822, fs:885-929) without scoring every window in float64
// ------------------------------------------------------------------------------------------------
// The greedy update takes the head of `background entries ++ candidates` sorted by PWMS (stable): only the best
// candidate matters, i.e. the FIRST window whose log2 score is the largest, if that exceeds the cut-off. The ranking
// pass of the SiteSampler finds the first window with the largest float64 PRODUCT. The two agree unless another
// window's product is so close to the maximum that both round to the same log2; every window that close lies in a
// chunk the ranking pass re-scores anyway, so the check is a comparison there, and such a case (or anything else the
// ranking pass cannot decide) falls back to the all-windows candidate list below.
// Inverse-CDF selection with a warp prefix sum, exact by construction. The reference walks the list and takes the
// first item whose float64 running sum reaches the pick (fs:746-754); that running sum is order-dependent, so a
// parallel scan cannot reproduce its bits -- but it can locate the bucket: scan and walk differ by at most
// (items + 64) * 2^-52 of the total mass, so when the pick is farther than four times that from both edges of the
// bucket the scan found, the walk must stop in the same bucket. Otherwise (probability ~1e-11 per pick), or when an
// item is negative (a cut-off below 0 admits negative PWMS; the walk's condition is then not monotone), the exact
// sequential walk runs. Lanes take contiguous blocks of the list, so lane order is list order.
__device__ __forceinline__ bool motif_roulette(const double *g, double gsum, int W, const double *cand_l, const int32_t *cand_w,
                                               int n_cand, double pick, int lane, double &pwms_out, int &site_out,
                                               bool scan_ok = true) {
    if (!scan_ok) return motif_roulette_exact(g, gsum, W, cand_l, cand_w, n_cand, pick, lane, pwms_out, site_out);
    const int total = W + n_cand;
    const int B = (total + 31) >> 5;
    const int i0 = min(total, lane * B), i1 = min(total, i0 + B);
    auto item = [&](int i) { return i < W ? g[i] : cand_l[i - W]; };
    double part = 0.0;
    bool negative = false;
    for (int i = i0; i < i1; ++i) {
        const double v = item(i);
        negative |= !(v >= 0.0);
        part += v;
    }
    double incl = part; // inclusive scan of the block sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    const double sum = __shfl_sync(FULL, incl, 31);
    bool decided = false;
    if (!__ballot_sync(FULL, negative) && sum > 0.0 && sum < INFINITY) {
        const double eps = 4.0 * (double)(total + 64) * 0x1p-52;
        const double target = pick * sum;                    // pick <= prefix / sum  <=>  pick * sum <= prefix (up to eps)
        const double before = incl - part;
        const unsigned holds = __ballot_sync(FULL, i0 < i1 && target <= incl); // first lane whose block reaches the pick
        if (holds) {
            const int src = __ffs(holds) - 1;
            int idx = -1;
            double lo = 0.0, hi = 0.0;
            if (lane == src) {
                double acc = before;
                for (int i = i0; i < i1; ++i) {
                    const double nxt = acc + item(i);
                    if (target <= nxt) {
                        idx = i;
                        lo = acc;
                        hi = nxt;
                        break;
                    }
                    acc = nxt;
                }
            }
            idx = __shfl_sync(FULL, idx, src);
            lo = __shfl_sync(FULL, lo, src);
            hi = __shfl_sync(FULL, hi, src);
            const double tol = eps * sum;
            // clear of both edges: lo + tol < target < hi - tol (idx = 0: the walk's lower edge is exactly 0, and a pick
            // below it makes the reference throw, so the exact walk decides that)
            if (idx >= 0 && target < hi - tol && (idx == 0 ? pick >= 0.0 : target > lo + tol)) {
                if (idx < W) {
                    pwms_out = g[idx];
                    site_out = -1;
                } else {
                    pwms_out = cand_l[idx - W];
                    site_out = cand_w[idx - W];
                }
                decided = true;
            }
        }
    }
    if (decided) return true;
    return motif_roulette_exact(g, gsum, W, cand_l, cand_w, n_cand, pick, lane, pwms_out, site_out);
}

template <int KP, int CH>
__device__ __forceinline__ bool pick_unique_argmax_ch(const WarpTables &T, const uint32_t *row, int W, int k, int lane,
                                                      double &hv_out, int &w_out) {
    using G = ScanGeom<KP, CH>;
    int32_t M1, M2;
    int S1;
    scan_fast<KP, CH>(row, W, T.ptab, lane, M1, M2, S1);
    const int32_t M = __reduce_max_sync(FULL, M1);
    const int32_t thr = M - (((k + 1) << KEY_IDX_BITS) + 255);
    if (__ballot_sync(FULL, M2 >= thr)) return false;
    unsigned cand = __ballot_sync(FULL, M1 >= thr);
    double p = 0.0, p2 = 0.0; // this lane's best and second-best re-scored window
    int w = INT32_MAX;
    while (cand) {
        const int src = __ffs(cand) - 1;
        cand &= cand - 1;
        const int32_t key = __shfl_sync(FULL, M1, src);
        const int seg = __shfl_sync(FULL, S1, src);
        const int wi = chunk_base<CH>(seg * G::CPS + src + 32 * (255 - (key & 255)), W) + lane;
        if (lane < CH && wi < W) {
            const double pi = exact_window<KP>(row, wi, k, T.wcol);
            if (better(pi, wi, p, w)) {
                p2 = fmax(p2, p);
                p = pi;
                w = wi;
            } else if (wi != w) {
                p2 = fmax(p2, pi);
            }
        }
    }
    double pm = p;
    int wm = w;
    warp_argmax(pm, wm);
    const double lim = pm * (1.0 - 1e-12); // log2 of anything below this differs from log2(pm) by > 1000 ulp
    const bool close = (w != wm && p >= lim) || p2 >= lim; // (pm = 0: every lane reports close -> fall back)
    if (__ballot_sync(FULL, close)) return false;
    hv_out = pm;
    w_out = wm;
    return true;
}

template <int KP>
__device__ __forceinline__ bool pick_unique_argmax(const WarpTables &T, const uint32_t *row, int W, int k, int lane, double &hv_out,
                                                   int &w_out) {
    if (W > 256) return pick_unique_argmax_ch<KP, 16>(T, row, W, k, lane, hv_out, w_out);
    if (W > 128) return pick_unique_argmax_ch<KP, 8>(T, row, W, k, lane, hv_out, w_out);
    return pick_unique_argmax_ch<KP, 4>(T, row, W, k, lane, hv_out, w_out);
}

// fixed-point log2 tables of an odds table built on the fly (data-derived background): what wtab_kernel precomputes
// for the fixed background. T.wcol holds the float64 odds (dummy column of an odd k = 1.0).
template <int KP>
__device__ __forceinline__ void fixed_point_tables(const WarpTables &T, int lane) {
    for (int e = lane; e < 8 * KP; e += 32) {
        double units = rint(log2(T.wcol[e]) * (double)(1 << LG_FRAC_BITS));
        units = fmin(fmax(units, -4000000.0), 4000000.0);
        T.lgcol[e] = (int)units * (1 << KEY_IDX_BITS);
    }
    __syncwarp();
    for (int idx = lane; idx < 16 * KP; idx += 32) {
        const int p = idx >> 4, nib = idx & 15;
        T.ptab[idx] = T.lgcol[(2 * p) * 4 + (nib & 3)] + T.lgcol[(2 * p + 1) * 4 + (nib >> 2)];
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// the MotifSampler kernel: one team (CTA of T warps) = one restart (fs:876-879 / fs:1034-1038)
// ------------------------------------------------------------------------------------------------
// Same division of labour as chain_kernel: one warp performs one whole site update, the T warps of a team work on T
// consecutive held-out sequences at once (a round).
//   stochastic sweep (fs:828-853 / fs:935-970): every n reads the INPUT state -- its own entry plus the all-sites
//     counts taken before the sweep -- so all N updates are independent and every result commits;
//   greedy sweeps (fs:788-822 / fs:885-929) are in place: speculative rounds as in chain_kernel -- results commit in
//     order up to and including the first warp whose accepted update changes the sites (moves, drops or gains a site).
// Per warp: candidate scratch (and, data-derived background, the background window products) in global memory.
#ifndef GIBBS_MOTIF_T4_BLOCKS
#define GIBBS_MOTIF_T4_BLOCKS 7 // 72 registers: all 1024 chains of a C2 step resident at once (5 blocks / 96 registers: 1.4 waves)
#endif
constexpr int MOTIF_BSUM_OFFSET = 2144; // 4 ints in the slack of the team's fixed shared memory (TEAM_FIXED_BYTES = 2176)

// MASKED = the set holds symbols outside A,C,G,T (a.s.mask != null): a separate instantiation, like chain_kernel's. Such a
// symbol is counted in a dead row when it lies inside a site (fs:211-215), a window over one scores 0 and its
// background-only probability is 0 (the pcv of a symbol outside the alphabet, fs:115-119); the held-out sequence's own
// such symbols enter the denominator of the data-derived background (fs:953 adds every symbol, fs:117 sums all 49 slots).
// Straggler hand-over as in chain_kernel: restarts need 5 to 20+ greedy sweeps, so once few of them are still running they
// pause at a sweep boundary (phase and sweep count in a.resume, the chain in a.pending_out) and the next launch on the
// stream continues them with teams of 8, then 16 warps. Scratch lists are indexed by CTA, not by chain.
template <int KP, int T, bool MASKED = false>
__global__ void __launch_bounds__(32 * T, (T == 1 ? 8 : T == 4 ? GIBBS_MOTIF_T4_BLOCKS : T == 8 ? 2 : 1)) motif_kernel(const MotifArgs m) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int THREADS = 32 * T;
    constexpr int R = (2 * T < 4) ? 4 : 2 * T;
    const ChainArgs &a = m.c;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int chain = blockIdx.x;
    if (a.from_list) { // continuing paused restarts: one CTA per list entry
        if ((int)blockIdx.x >= *a.pending_in_n) return;
        chain = a.pending_in[blockIdx.x];
    }
    const TeamSmem S = carve_smem(smem_raw, T);
    const WarpTables WT = warp_tables(S, warp);
    require_aligned_tables(WT);
    int32_t *bsum = reinterpret_cast<int32_t *>(smem_raw + MOTIF_BSUM_OFFSET); // data background: base counts over the sequences that have a site
    const int N = a.s.n, k = a.k;
    int32_t *sites = a.sites + (size_t)chain * N;
    double *pw = a.scores + (size_t)chain * N; // PWMS of the MotifIndex state
    double *hv = a.hv + (size_t)chain * N;
    double *cand_l = m.cand_l + ((size_t)blockIdx.x * T + warp) * m.bg.wstride;
    int32_t *cand_w = m.cand_w + ((size_t)blockIdx.x * T + warp) * m.bg.wstride;
    double *gbuf = m.data_bg ? m.gbuf + ((size_t)blockIdx.x * T + warp) * m.bg.wstride : nullptr;
    const uint64_t chain_uid = (uint64_t)a.chain_id_base + (uint64_t)chain;
    const double raw_gate = exp2(a.cutoff) * (1.0 - 0x1p-30);

    RowRing<R> ring;
    ring.init(S, a.s, 0, tid);
    if (tid < 16) S.lut[tid] = hist_lut_entry(tid);
    team_sync<T>();
    if (warp == 0) ring.fill_span(0u, 0, R, lane);

    unsigned long long st_updates = 0, st_windows = 0, st_slow = 0, st_spec = 0; // st_slow: updates that scored every window in float64
    int st_sweeps = 0, capped = 0;
    uint32_t vbase = 0;

    if (m.init_done && !a.from_list) { // the random starts ran in their own kernel (gibbs_api.cu, launch_random_starts): the state is
        // SiteSampler.getPWMOfRandomStarts[WithBPV] |> createMotifIndex prob [position] (fs:876-877, fs:993-994)
        for (int n = tid; n < N; n += THREADS) pw[n] = log2_ref(__ldcg(hv + n));
        team_sync<T>();
    }
    int phase = MPH_STOCH;
    while (phase < MPH_DONE && !((a.phase_mask >> (phase == MPH_STOCH ? 4 : 5)) & 1)) ++phase;
    int sweeps_in_phase = 0;
    bool resumed = false, paused = false;
    if (a.from_list) {
        const int r = a.resume[chain]; // phase | capped so far << 7 | sweeps in phase << 8
        phase = r & 127;
        capped = (r >> 7) & 1;
        sweeps_in_phase = r >> 8;
        resumed = true;
    }
    while (phase != MPH_DONE) {
        if (phase == MPH_STOCH || sweeps_in_phase == 0 || resumed) {
            resumed = false;
            site_counts<KP, T>(a.s, sites, -1, k, SHIFT_NONE, S.total, S.lut, S.fix, tid);
            if (m.data_bg) {
                if (tid < 4) bsum[tid] = 0;
                team_sync<T>();
                int part[4] = {0, 0, 0, 0};
                for (int i = tid; i < N; i += THREADS)
                    if (__ldcg(sites + i) >= 0) {
#pragma unroll
                        for (int b = 0; b < 4; ++b) part[b] += __ldg(m.basecnt + i * 4 + b);
                    }
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int s = __reduce_add_sync(FULL, part[b]);
                    if (lane == 0 && s != 0) atomicAdd(&bsum[b], s);
                }
                team_sync<T>();
            }
        } else {
            team_sync<T>(); // the previous sweep's last round wrote sites / pw after its only barrier
        }
        bool changed = false;
        int n0 = 0;
        // greedy: speculation width adapts as in chain_kernel. The first GIBBS_MOTIF_NARROW_SWEEPS greedy sweeps move a site in
        // most updates: their rounds start at width 1 and narrow after a discard. Later sweeps never narrow: they discard
        // little, and a round that stays wide costs the other restarts of the SM less than it gains.
        const int min_w = (phase == MPH_GREEDY && sweeps_in_phase < GIBBS_MOTIF_NARROW_SWEEPS) ? 1 : T;
        int width = (phase == MPH_GREEDY) ? min_w : T;
        unsigned round = 0;
        while (n0 < N) {
            const int n = n0 + warp;
            const bool active = n < N && warp < width;
            int flag = 0, site_n = -1, new_site = -1, W = 0;
            double new_pw = 0.0;
            bool has_own = false;
            uint64_t own = 0, neu = 0;
            int cn[4] = {0, 0, 0, 0};
            int masked_n = -1;
            uint64_t own_mk = 0;
            if (active) {
                const uint32_t *row = ring.wait(vbase + (uint32_t)n);
                W = __ldg(a.s.len + n) - k + 1;
                {
                    site_n = __ldcg(sites + n);
                    const double pw_n = __ldcg(pw + n);
                    has_own = site_n >= 0;
                    own = has_own ? kmer_shared<KP>(row, site_n) : 0;
                    if (MASKED && __ldg(a.s.rowflag + n) != 0) {
                        masked_n = n;
                        if (has_own) own_mk = mask_kmer(a.s.mask, a.s.row_words, n, site_n, k);
                    }
                    const double *g_n = m.bg.g + (size_t)n * m.bg.wstride;
                    double gsum_n = 0.0, gmax_n = 0.0;
                    if (!m.data_bg) {
                        if (MASKED && own_mk != 0) build_tables_masked<KP>(WT, S.total, own, k, a.wtab, lane, own_mk);
                        else build_tables<KP>(WT, S.total, has_own, own, k, a.wtab, lane);
                        gsum_n = __ldg(m.bg.gsum + n);
                        gmax_n = __ldg(m.bg.gmax + n);
                    } else {
                        // background of this held-out sequence (fs:896-905): the OTHER sequences that have a site, outside
                        // those sites (fused over the alphabet), plus every base of the held-out sequence
                        for (int e = lane; e < 4 * k; e += 32) {
                            int c = S.total[e];
                            if (has_own && (int)((own >> (2 * (e >> 2))) & 3u) == (e & 3) && !(MASKED && ((own_mk >> (2 * (e >> 2))) & 1u))) c -= 1;
                            WT.lgcol[e] = c;
                        }
                        __syncwarp();
                        int F[4], fs = 0;
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            int s = 0;
                            for (int j = lane; j < k; j += 32) s += WT.lgcol[j * 4 + b];
                            cn[b] = __ldg(m.basecnt + n * 4 + b);
                            F[b] = bsum[b] - (has_own ? cn[b] : 0) - __reduce_add_sync(FULL, s) + cn[b];
                            fs += F[b];
                        }
                        if (MASKED && masked_n >= 0) fs += __ldg(a.maskcnt + n); // its own symbols outside the alphabet (fs:953, fs:117)
                        const double den = __dadd_rn((double)fs, m.alpha_pc);
                        double q[4];
#pragma unroll
                        for (int b = 0; b < 4; ++b) q[b] = __ddiv_rn(__dadd_rn((double)F[b], m.pc), den); // fs:119
                        for (int e = lane; e < 8 * KP; e += 32) { // PWM = PPM / pcv (fs:286); dummy column of an odd k = 1.0
                            const int b = e & 3;
                            const double qb = b == 0 ? q[0] : b == 1 ? q[1] : b == 2 ? q[2] : q[3];
                            WT.wcol[e] = (e >> 2) < k ? __ddiv_rn(__ldg(m.pvals + WT.lgcol[e]), qb) : 1.0;
                        }
                        // background-only probability of every window (fs:776), first maximum, and their sum in list order:
                        // the same left-to-right product as a window score, over a table whose every column is q
                        // (kept in the pair-table space, which is rebuilt after this loop when the greedy ranking pass runs)
                        double *qtab = reinterpret_cast<double *>(WT.ptab);
                        for (int e = lane; e < 8 * KP; e += 32) {
                            const int b = e & 3;
                            qtab[e] = (e >> 2) < k ? (b == 0 ? q[0] : b == 1 ? q[1] : b == 2 ? q[2] : q[3]) : 1.0;
                        }
                        __syncwarp();
                        const uint8_t *seq_n = nullptr;
                        if (MASKED && masked_n >= 0) { // symbol counts of the held-out sequence (candidate scratch is free here)
                            seq_n = m.ascii + __ldg(m.off + n);
                            for (int e = lane; e < 64; e += 32) cand_w[e] = 0;
                            __syncwarp();
                            for (int i = lane; i < W + k - 1; i += 32) atomicAdd(&cand_w[seq_n[i] - 42], 1);
                            __syncwarp();
                        }
                        double bestg = 0.0;
                        for (int w0 = 0; w0 < W; w0 += 32) {
                            const int w = w0 + lane;
                            if (w < W) {
                                double v = exact_window<KP>(row, w, k, qtab);
                                if (MASKED && masked_n >= 0 && mask_kmer(a.s.mask, a.s.row_words, n, w, k) != 0)
                                    v = masked_background_window(seq_n, w, k, q, cand_w);
                                gbuf[w] = v;
                                bestg = fmax(bestg, v);
                            }
                        }
                        __syncwarp();
                        {
                            const uint32_t hi = (uint32_t)__double2hiint(bestg), mh = __reduce_max_sync(FULL, hi);
                            const uint32_t lo = (hi == mh) ? (uint32_t)__double2loint(bestg) : 0u, ml = __reduce_max_sync(FULL, lo);
                            gmax_n = __hiloint2double((int)mh, (int)ml);
                        }
                        if (phase == MPH_STOCH) { // List.sum visits the background entries first, in window order (fs:748)
                            for (int w0 = 0; w0 < W; w0 += 32) {
                                const double v = (w0 + lane < W) ? gbuf[w0 + lane] : 0.0;
                                const int lim = min(32, W - w0);
                                for (int j = 0; j < lim; ++j) gsum_n = __dadd_rn(gsum_n, __shfl_sync(FULL, v, j));
                            }
                        }
                        g_n = gbuf;
                    }
                    double best_l;
                    int best_w;
                    int n_cand = -1;
                    bool slow = false;
                    if (phase == MPH_GREEDY && m.greedy_fast_ok && !(MASKED && masked_n >= 0)) { // only the best candidate matters: rank, re-score, compare
                        if (m.data_bg) fixed_point_tables<KP>(WT, lane);
                        double pbest;
                        if (pick_unique_argmax<KP>(WT, row, W, k, lane, pbest, best_w)) {
                            best_l = log2_ref(pbest);
                            n_cand = best_l > a.cutoff ? 1 : 0; // fs:735
                        }
                    }
                    int gated = -1;
                    if (n_cand < 0) {
                        gated = motif_gate<KP, MASKED>(WT, row, W, k, raw_gate, cand_l, cand_w, lane, &a.s, masked_n);
                        if (phase != MPH_STOCH || !m.roulette_scan_ok) {
                            n_cand = motif_logs(a.cutoff, cand_l, cand_w, gated, lane, best_l, best_w);
                            gated = -1;
                        }
                        slow = true;
                    }
                    bool take;
                    if (phase == MPH_STOCH) { // fs:828-853: one uniform per n, every n reads the input state
                        const uint64_t d = (uint64_t)N * (uint64_t)(N - 1) + (uint64_t)n;
                        double u;
                        if (a.rng_mode == 0) {
                            const uint64_t blk = d >> 2;
                            const uint4 r = philox4x32_10(
                                make_uint4((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)chain_uid, (uint32_t)(chain_uid >> 32)),
                                make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
                            const uint32_t word = (d & 3) == 0 ? r.x : (d & 3) == 1 ? r.y : (d & 3) == 2 ? r.z : r.w;
                            u = (double)word * (1.0 / 4294967296.0);
                        } else {
                            u = ((int64_t)d < a.uniforms_per_chain) ? __ldg(a.uniforms + (size_t)chain * a.uniforms_per_chain + d) : 0.0;
                        }
                        bool ok = gated >= 0 && motif_stoch_fast(gsum_n, a.cutoff, cand_l, cand_w, gated, u, lane, new_pw, new_site);
                        if (!ok) {
                            if (gated >= 0) n_cand = motif_logs(a.cutoff, cand_l, cand_w, gated, lane, best_l, best_w);
                            ok = motif_roulette(g_n, gsum_n, W, cand_l, cand_w, n_cand, u, lane, new_pw, new_site,
                                                m.roulette_scan_ok != 0);
                        }
                        if (!ok) {
                            if (lane == 0) atomicExch(m.error, 1);
                            new_pw = pw_n;
                            new_site = site_n;
                        }
                        take = true;
                    } else { // fs:788-822: first maximum by PWMS over background entries ++ candidates
                        if (n_cand > 0 && best_l > gmax_n) {
                            new_pw = best_l;
                            new_site = best_w;
                        } else {
                            new_pw = gmax_n;
                            new_site = -1;
                        }
                        take = new_pw > pw_n; // fs:816
                    }
                    const bool moved = take && phase == MPH_GREEDY && new_site != site_n;
                    if (moved && new_site >= 0) neu = kmer_shared<KP>(row, new_site); // rows are not read after the sync
                    flag = (take ? 1 : 0) | (moved ? 2 : 0) | (slow ? 4 : 0);
                }
            }
            int32_t *flags = S.flags + (round & 1) * T; // double-buffered: one team sync per round suffices
            ++round;
            if (lane == 0) flags[warp] = flag;
            team_sync<T>();
            // greedy only: warps after the first mover of the round saw stale counts
            const unsigned movers = __ballot_sync(FULL, lane < T && (flags[lane < T ? lane : 0] & 2) != 0);
            const int first_mover = movers ? __ffs(movers) - 1 : T; // (only greedy updates set the mover bit)
            const int last_commit = min(first_mover, width - 1);
            changed |= movers != 0;
            if (active) {
                if (warp <= last_commit) {
                    st_updates += 1;
                    st_windows += (unsigned long long)W;
                    st_slow += (flag & 4) ? 1 : 0;
                    if ((flag & 1) && lane == 0) {
                        sites[n] = new_site;
                        pw[n] = new_pw;
                    }
                } else {
                    st_spec += 1;
                }
            }
            const int committed = min(last_commit + 1, N - n0);
            if (warp == 0) ring.fill_span(vbase + (uint32_t)(n0 + R), n0 + R, committed, lane); // their rows are free
            n0 += committed;
            if (phase == MPH_GREEDY) {
                if (first_mover < T) { // in-place sweep: later n see the new state (fs:795 reads acc): -old k-mer, +new k-mer
                    if (warp == first_mover) {
                        uint64_t neu_mk = 0;
                        if (MASKED && masked_n >= 0 && new_site >= 0) neu_mk = mask_kmer(a.s.mask, a.s.row_words, n, new_site, k);
                        if (lane < k) { // (bases outside A,C,G,T were never counted)
                            if (has_own && !(MASKED && ((own_mk >> (2 * lane)) & 1u))) S.total[lane * 4 + (int)((own >> (2 * lane)) & 3u)] -= 1;
                            if (new_site >= 0 && !(MASKED && ((neu_mk >> (2 * lane)) & 1u))) S.total[lane * 4 + (int)((neu >> (2 * lane)) & 3u)] += 1;
                        }
                        if (m.data_bg && has_own != (new_site >= 0) && lane < 4) { // the sequence gained or lost its site
                            const int d = lane == 0 ? cn[0] : lane == 1 ? cn[1] : lane == 2 ? cn[2] : cn[3];
                            bsum[lane] += new_site >= 0 ? d : -d;
                        }
                    }
                    team_sync<T>(); // counts updated before the next round builds its tables
                    width = max(min_w, width >> 1);
                } else {
                    width = min(T, width * 2);
                }
            }
        }
        vbase += (uint32_t)N;
        st_sweeps += 1;
        bool next = true;
        if (phase == MPH_GREEDY) {
            ++sweeps_in_phase;
            next = !changed; // Positions(acc) = Positions(bestMotif), fs:791
            if (!next && sweeps_in_phase >= a.max_sweeps) {
                next = true;
                capped = 1;
            }
        }
        if (next) {
            sweeps_in_phase = 0;
            ++phase;
            while (phase < MPH_DONE && !((a.phase_mask >> (phase == MPH_STOCH ? 4 : 5)) & 1)) ++phase;
        }
        // sweep boundary: when few restarts are still running, hand this one over to the wide-team launch
        if (phase != MPH_DONE && a.pause_below > 0) {
            if (tid == 0) S.flags[2 * T] = (*(volatile int32_t *)a.active <= a.pause_below && st_sweeps >= a.pause_min_sweeps) ? 1 : 0;
            team_sync<T>();
            if (S.flags[2 * T]) {
                paused = true;
                break;
            }
        }
    }
    if (tid == 0) // the ring always has R rows in flight: let them land before the CTA exits
        for (int i = 0; i < R; ++i) ring.wait(vbase + (uint32_t)i);
    team_sync<T>();
    if (!paused)
        for (int n = tid; n < N; n += THREADS) hv[n] = __ldcg(pw + n);
    if (lane == 0) {
        atomicAdd(a.stats + ST_SITE_UPDATES, st_updates);
        atomicAdd(a.stats + ST_EXACT_RESCANS, st_slow);
        atomicAdd(a.stats + ST_WINDOW_SCORES, st_windows);
        atomicAdd(a.stats + ST_SPECULATED, st_spec);
    }
    if (tid == 0) {
        atomicAdd(a.stats + ST_SWEEPS, (unsigned long long)st_sweeps);
        if (!paused) atomicAdd(a.stats + ST_CAPPED, (unsigned long long)capped); // (a restart counts once, where it ends)
        if (paused) {
            a.resume[chain] = phase | (capped << 7) | (sweeps_in_phase << 8);
            a.pending_out[atomicAdd(a.pending_out_n, 1)] = chain;
        } else {
            double sum = 0.0;
            for (int n = 0; n < N; ++n) sum = __dadd_rn(sum, __ldcg(pw + n));
            a.sums[chain] = sum;
            if (a.active) atomicSub(a.active, 1);
        }
    }
}

// primitive: candidate list + one roulette pick for a given state (gibbs_pick_roulette)
struct RouletteArgs {
    PrimArgs p;
    BgTables bg;
    double cutoff;
    double u;
    double *cand_l;
    int32_t *cand_w;
    double *pwms_out;
    int32_t *site_out; // [2]: site, ok flag
};

template <int KP>
static __global__ void __launch_bounds__(32) roulette_kernel(const RouletteArgs r) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const PrimArgs &a = r.p;
    const int lane = threadIdx.x;
    const TeamSmem S = carve_smem(smem_raw, 1);
    const WarpTables WT = warp_tables(S, 0);
    RowRing<4> ring;
    ring.init(S, a.s, a.heldout, lane);
    if (lane < 16) S.lut[lane] = hist_lut_entry(lane);
    __syncwarp();
    if (lane == 0) ring.fill(1);
    site_counts<KP, 1>(a.s, a.sites, a.heldout, a.k, SHIFT_NONE, S.total, S.lut, S.fix, lane);
    const uint32_t *row = ring.wait(0);
    build_tables<KP>(WT, S.total, false, 0, a.k, a.wtab, lane);
    const int W = __ldg(a.s.len + a.heldout) - a.k + 1;
    double best_l;
    int best_w;
    const int n_cand = motif_candidates<KP, true>(WT, row, W, a.k, r.cutoff, exp2(r.cutoff) * (1.0 - 0x1p-30), r.cand_l, r.cand_w,
                                                  lane, best_l, best_w, &a.s, row_masked(a.s, a.heldout) ? a.heldout : -1);
    double pwms = 0.0;
    int site = -1;
    const bool ok = motif_roulette(r.bg.g + (size_t)a.heldout * r.bg.wstride, __ldg(r.bg.gsum + a.heldout), W, r.cand_l,
                                   r.cand_w, n_cand, r.u, lane, pwms, site);
    if (lane == 0) {
        *r.pwms_out = pwms;
        r.site_out[0] = site;
        r.site_out[1] = ok ? 1 : 0;
    }
}

} // namespace gibbs
