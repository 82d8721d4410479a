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
        double s = w < W ? exact_window<KP>(row, w, T.wcol) : 0.0;
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
            const double pi = exact_window<KP>(row, wi, T.wcol);
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
#include "gibbs_motif_body.inc"
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
