// gibbssampling_b200/csrc/gibbs_drift_dev.cuh -- device routines of the data-derived (drifting) background
// (getBestPWMSs fs:462-479): the all-windows float64 scan and the float32 ranking pass with exact re-scoring.
// Used by chain_kernel<.., DRIFT = true> (SiteSampler, gibbs_drift_launch.cu) and by motif_kernel (random starts).
#pragma once
#include "gibbs_device.cuh"

namespace gibbs {

__device__ __forceinline__ int base_at(const uint32_t *row, int pos) { return (row[pos >> 4] >> ((pos & 15) * 2)) & 3; }

// getBestPWMSs (fs:462-479) for the staged row. ppm = smem [k][4] float64 PPM of the leave-one-out counts.
// f0[b] = fused background counts of the others; cn[b] = base counts of this sequence; f0g = f0[Gap] when Gap is a
// member of the alphabet (else 0): a row without Gap still has it in every denominator (fs:116 sums every slot).
__device__ __forceinline__ void scan_drifting(const uint32_t *row, int W, int k, const double *ppm, const int *f0,
                                              const int *cn, int f0g, double pc, double alpha_pc, int lane, double &hv_out,
                                              int &w_out) {
    const int B = (W + 31) >> 5;
    const int w_begin = min(W, lane * B), w_end = min(W, w_begin + B);
    // pass A: occurrences summed over this lane's windows (sliding counts, 4 byte fields: k <= 32)
    int blocksum[4] = {0, 0, 0, 0};
    if (w_begin < w_end) {
        uint32_t occ = 0;
        for (int j = 0; j < k; ++j) occ += 1u << (8 * base_at(row, w_begin + j));
        for (int w = w_begin; w < w_end; ++w) {
#pragma unroll
            for (int b = 0; b < 4; ++b) blocksum[b] += (int)((occ >> (8 * b)) & 255u);
            if (w + 1 < w_end) {
                occ -= 1u << (8 * base_at(row, w));
                occ += 1u << (8 * base_at(row, w + k));
            }
        }
    }
    // exclusive prefix over lanes
    int before[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        int v = blocksum[b];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, v, o);
            if (lane >= o) v += t;
        }
        before[b] = v - blocksum[b];
    }
    // pass B: every window exactly
    double hv = 0.0;
    int hw = 0;
    if (w_begin < w_end) {
        int run[4];
#pragma unroll
        for (int b = 0; b < 4; ++b) run[b] = before[b];
        uint32_t oc = 0;
        for (int j = 0; j < k; ++j) oc += 1u << (8 * base_at(row, w_begin + j));
        for (int w = w_begin; w < w_end; ++w) {
            int F[4], sum = f0g;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                run[b] += (int)((oc >> (8 * b)) & 255u);
                F[b] = f0[b] + (w + 1) * cn[b] - run[b];
                sum += F[b];
            }
            const double den = __dadd_rn((double)sum, alpha_pc);                       // fs:117
            double pcv[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) pcv[b] = __ddiv_rn(__dadd_rn((double)F[b], pc), den); // fs:119
            double v = 1.0;
            for (int j = 0; j < k; ++j) {
                const int b = base_at(row, w + j);
                const double q = b == 0 ? pcv[0] : b == 1 ? pcv[1] : b == 2 ? pcv[2] : pcv[3];
                v = __dmul_rn(v, __ddiv_rn(ppm[j * 4 + b], q));                           // fs:286, fs:292
            }
            if (v > hv) {
                hv = v;
                hw = w;
            }
            if (w + 1 < w_end) {
                oc -= 1u << (8 * base_at(row, w));
                oc += 1u << (8 * base_at(row, w + k));
            }
        }
    }
    warp_argmax(hv, hw);
    hv_out = hv;
    w_out = hw;
}

// ------------------------------------------------------------------------------------------------
// ranking pass for the drifting background
// ------------------------------------------------------------------------------------------------
// log2 score(w) = sum_j log2 ppm[j][b_j] - sum_b occ_w[b] log2(F_w[b] + pc) + k log2(den_w): the first sum comes from
// a float32 pair table (two bases per lookup), the rest from 5 MUFU.LG2 per window. The float32 value is within
// ~1.2e-3 of the true log2 score (k <= 32: table entries and MUFU.LG2 are good to 2 ulp of values < 32, sums stay below
// 1024 where a float32 ulp is 6.1e-5), so the float64 argmax lies among the windows within DRIFT_MARGIN of the float32
// maximum. Those windows (at most one per lane, else the exact scan runs) are re-scored exactly as scan_drifting does.
constexpr float DRIFT_MARGIN = 0.03125f;

// MUFU.LG2 alone: the arguments of the ranking pass are normal floats (counts + pc with pc >= 1e-30, checked on the
// host), so the denormal rescaling that __log2f wraps around the instruction is dead weight (4 of 5 instructions)
__device__ __forceinline__ float lg2_normal(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// float32 log2 of the PPM in pair-table form: pt[p*16 + nib] = lg[2p][nib & 3] + lg[2p+1][nib >> 2]
template <int KP>
__device__ __forceinline__ void drift_pair_table(const double *ppm, float *lg, float *pt, int k, int lane) {
    for (int e = lane; e < 8 * KP; e += 32) lg[e] = (e < 4 * k) ? __log2f((float)ppm[e]) : 0.0f;
    __syncwarp();
    for (int idx = lane; idx < 16 * KP; idx += 32) {
        const int p = idx >> 4, nib = idx & 15;
        pt[idx] = lg[(2 * p) * 4 + (nib & 3)] + lg[(2 * p + 1) * 4 + (nib >> 2)];
    }
    __syncwarp();
}

// one window exactly, the body of scan_drifting's pass B (fs:471-474, fs:290-293)
__device__ __forceinline__ double drift_exact_window(const uint32_t *row, int w, int k, const double *ppm, const int *f0,
                                                     const int *cn, const int *run, double pc, double alpha_pc) {
    int F[4], sum = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        F[b] = f0[b] + (w + 1) * cn[b] - run[b];
        sum += F[b];
    }
    const double den = __dadd_rn((double)sum, alpha_pc);
    double pcv[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) pcv[b] = __ddiv_rn(__dadd_rn((double)F[b], pc), den);
    double v = 1.0;
    for (int j = 0; j < k; ++j) {
        const int b = base_at(row, w + j);
        const double q = b == 0 ? pcv[0] : b == 1 ? pcv[1] : b == 2 ? pcv[2] : pcv[3];
        v = __dmul_rn(v, __ddiv_rn(ppm[j * 4 + b], q));
    }
    return v;
}

// Returns false when the exact scan has to run instead (a lane with two windows inside the margin).
template <int KP>
__device__ __forceinline__ bool scan_drifting_fast(const uint32_t *row, int W, int k, const double *ppm, const float *pt,
                                                   const int *f0, const int *cn, int f0g, double pc, double alpha_pc, int lane,
                                                   double &hv_out, int &w_out) {
    const int B = (W + 31) >> 5;
    const int w_begin = min(W, lane * B), w_end = min(W, w_begin + B);
    int blocksum[4] = {0, 0, 0, 0};
    if (w_begin < w_end) { // occurrences summed over this lane's windows (as scan_drifting's pass A)
        uint32_t occ = 0;
        for (int j = 0; j < k; ++j) occ += 1u << (8 * base_at(row, w_begin + j));
        for (int w = w_begin; w < w_end; ++w) {
#pragma unroll
            for (int b = 0; b < 4; ++b) blocksum[b] += (int)((occ >> (8 * b)) & 255u);
            if (w + 1 < w_end) {
                occ -= 1u << (8 * base_at(row, w));
                occ += 1u << (8 * base_at(row, w + k));
            }
        }
    }
    int run[4];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        int v = blocksum[b];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, v, o);
            if (lane >= o) v += t;
        }
        run[b] = v - blocksum[b];
    }
    const float ninf = __int_as_float(0xff800000);
    float M1 = ninf, M2 = ninf;
    int w1 = 0, run1[4] = {0, 0, 0, 0};
    if (w_begin < w_end) {
        const float pcf = (float)pc, apcf = (float)alpha_pc, kf = (float)k;
        uint32_t oc = 0;
        for (int j = 0; j < k; ++j) oc += 1u << (8 * base_at(row, w_begin + j));
        for (int w = w_begin; w < w_end; ++w) {
            float bg = 0.0f;
            int sum = f0g;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int ob = (int)((oc >> (8 * b)) & 255u);
                run[b] += ob;
                const int F = f0[b] + (w + 1) * cn[b] - run[b];
                sum += F;
                bg = fmaf((float)ob, lg2_normal((float)F + pcf), bg);
            }
            bg = fmaf(-kf, lg2_normal((float)sum + apcf), bg);
            const uint64_t kmer = kmer_shared<KP>(row, w);
            float mot = 0.0f;
#pragma unroll
            for (int p = 0; p < KP; ++p) mot += pt[p * 16 + ((uint32_t)(kmer >> (4 * p)) & 15u)];
            const float a = mot - bg;
            if (a > M1) {
                M2 = M1;
                M1 = a;
                w1 = w;
#pragma unroll
                for (int b = 0; b < 4; ++b) run1[b] = run[b];
            } else if (a > M2) {
                M2 = a;
            }
            if (w + 1 < w_end) { // slide: base w leaves, base w + k enters (both inside the 64 bits just fetched when k < 32)
                oc -= 1u << (8 * ((uint32_t)kmer & 3u));
                oc += 1u << (8 * (k < 32 ? (int)((uint32_t)(kmer >> (2 * k)) & 3u) : base_at(row, w + k)));
            }
        }
    }
    float M = M1;
#pragma unroll
    for (int o = 16; o; o >>= 1) M = fmaxf(M, __shfl_xor_sync(FULL, M, o));
    const float thr = M - DRIFT_MARGIN;
    if (__ballot_sync(FULL, M2 >= thr)) return false;
    // Candidates (normally one) are re-scored by the whole warp with the reference's own operations: lanes 0-3 divide
    // out the four background probabilities, lane j divides column j's ratio, and the product is taken left to right
    // (fs:290-293) with one shuffle + multiply per column -- 2 dependent divisions instead of k + 4.
    unsigned cand = __ballot_sync(FULL, M1 >= thr);
    double hv = 0.0;
    int hw = INT32_MAX;
    while (cand) {
        const int src = __ffs(cand) - 1;
        cand &= cand - 1;
        const int wc = __shfl_sync(FULL, w1, src);
        int F[4], sum = f0g;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            F[b] = f0[b] + (wc + 1) * cn[b] - __shfl_sync(FULL, run1[b], src);
            sum += F[b];
        }
        const double den = __dadd_rn((double)sum, alpha_pc);                       // fs:117
        const int fb = lane == 0 ? F[0] : lane == 1 ? F[1] : lane == 2 ? F[2] : F[3];
        const double q_lane = __ddiv_rn(__dadd_rn((double)fb, pc), den);             // fs:119, lanes 0-3 hold pcv[A,C,G,T]
        const int b = lane < k ? base_at(row, wc + lane) : 0;
        const double q = __shfl_sync(FULL, q_lane, b);
        const double ratio = lane < k ? __ddiv_rn(ppm[lane * 4 + b], q) : 1.0;       // fs:286
        double v = 1.0;
        for (int j = 0; j < k; ++j) v = __dmul_rn(v, __shfl_sync(FULL, ratio, j));   // fs:292
        if (better(v, wc, hv, hw)) { // largest product, lowest window on ties = the first strict maximum of fs:476
            hv = v;
            hw = wc;
        }
    }
    hv_out = hv;
    w_out = hw;
    return true;
}

// The same ranking pass over per-sequence PREFIX TABLES: ss[t][b] = sum_{u < t} (number of base b among the first u
// bases), a property of the sequence computed once (prefix_kernel). With P[t] = ss[t+1] - ss[t] the occurrences of a
// window are P[w+k] - P[w] and the drifting sum over the windows before it is
//   sum_{m <= w} occ_m = (ss[w+k+1] - ss[k]) - ss[w+1],
// so no sliding counters, no pass over the lane's windows to seed them, no cross-lane prefix, and lanes take
// interleaved windows (coalesced 16-byte table reads). Four loads and a dozen integer adds replace ~45 instructions
// per window and eight live registers.
template <int KP>
__device__ __forceinline__ bool scan_drifting_tables(const uint32_t *row, const int4 *__restrict__ ss, int W, int k, const double *ppm,
                                                     const float *pt, const int *f0, const int *cn, int f0g, double pc, double alpha_pc,
                                                     int lane, double &hv_out, int &w_out) {
    const float ninf = __int_as_float(0xff800000);
    const float pcf = (float)pc, apcf = (float)alpha_pc, kf = (float)k;
    const int4 sk = __ldg(ss + k);
    float M1 = ninf, M2 = ninf;
    int w1 = 0;
    for (int w = lane; w < W; w += 32) {
        const int4 a0 = __ldg(ss + w), a1 = __ldg(ss + w + 1), b0 = __ldg(ss + w + k), b1 = __ldg(ss + w + k + 1);
        const int occ[4] = {(b1.x - b0.x) - (a1.x - a0.x), (b1.y - b0.y) - (a1.y - a0.y), (b1.z - b0.z) - (a1.z - a0.z),
                            (b1.w - b0.w) - (a1.w - a0.w)};
        const int run[4] = {b1.x - sk.x - a1.x, b1.y - sk.y - a1.y, b1.z - sk.z - a1.z, b1.w - sk.w - a1.w};
        float bg = 0.0f;
        int sum = f0g;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int F = f0[b] + (w + 1) * cn[b] - run[b];
            sum += F;
            bg = fmaf((float)occ[b], lg2_normal((float)F + pcf), bg);
        }
        bg = fmaf(-kf, lg2_normal((float)sum + apcf), bg);
        const uint64_t kmer = kmer_shared<KP>(row, w);
        float mot = 0.0f;
#pragma unroll
        for (int p = 0; p < KP; ++p) mot += pt[p * 16 + ((uint32_t)(kmer >> (4 * p)) & 15u)];
        const float a = mot - bg;
        if (a > M1) {
            M2 = M1;
            M1 = a;
            w1 = w;
        } else if (a > M2) {
            M2 = a;
        }
    }
    float M = M1;
#pragma unroll
    for (int o = 16; o; o >>= 1) M = fmaxf(M, __shfl_xor_sync(FULL, M, o));
    const float thr = M - DRIFT_MARGIN;
    if (__ballot_sync(FULL, M2 >= thr)) return false;
    unsigned cand = __ballot_sync(FULL, M1 >= thr);
    double hv = 0.0;
    int hw = INT32_MAX;
    while (cand) { // cooperative re-scoring with the reference's own operations, as in scan_drifting_fast
        const int src = __ffs(cand) - 1;
        cand &= cand - 1;
        const int wc = __shfl_sync(FULL, w1, src);
        const int4 a1 = __ldg(ss + wc + 1), b1 = __ldg(ss + wc + k + 1);
        const int run[4] = {b1.x - sk.x - a1.x, b1.y - sk.y - a1.y, b1.z - sk.z - a1.z, b1.w - sk.w - a1.w};
        int F[4], sum = f0g;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            F[b] = f0[b] + (wc + 1) * cn[b] - run[b];
            sum += F[b];
        }
        const double den = __dadd_rn((double)sum, alpha_pc);                       // fs:117
        const int fb = lane == 0 ? F[0] : lane == 1 ? F[1] : lane == 2 ? F[2] : F[3];
        const double q_lane = __ddiv_rn(__dadd_rn((double)fb, pc), den);             // fs:119, lanes 0-3 hold pcv[A,C,G,T]
        const int b = lane < k ? base_at(row, wc + lane) : 0;
        const double q = __shfl_sync(FULL, q_lane, b);
        const double ratio = lane < k ? __ddiv_rn(ppm[lane * 4 + b], q) : 1.0;       // fs:286
        double v = 1.0;
        for (int j = 0; j < k; ++j) v = __dmul_rn(v, __shfl_sync(FULL, ratio, j));   // fs:292
        if (better(v, wc, hv, hw)) {
            hv = v;
            hw = wc;
        }
    }
    hv_out = hv;
    w_out = hw;
    return true;
}

// ------------------------------------------------------------------------------------------------
// the all-windows scan for a held-out sequence with symbols outside A,C,G,T (rare path, out of line)
// ------------------------------------------------------------------------------------------------
// Such a symbol is not in `alphabet`: its PWM row is 0, so a window that holds it scores 0 (fs:283-287). The drifting
// background still sees it: increaseInPlaceFCVOf adds EVERY symbol of the held-out sequence (fs:79-81, fs:471) and
// substractSegmentCountsFrom takes the window's symbols out again (fs:84-88), so the dead rows hold
// (w + 1) M_n - sum_{m <= w} occM_m (M_n = such symbols in the sequence, occM_m = in window m) and add to the
// denominator of createNormalizedPCVOfFCV, which sums all 49 slots (fs:116). The other sequences' dead rows were
// dropped by fuseFrequencyVectors (fs:67-69).
__device__ __forceinline__ int mask_at(const uint32_t *__restrict__ mrow, int pos) { return (__ldg(mrow + (pos >> 4)) >> ((pos & 15) * 2)) & 1; }
__device__ __forceinline__ int mask2_at(const uint32_t *__restrict__ mrow, int pos) { return (__ldg(mrow + (pos >> 4)) >> ((pos & 15) * 2)) & 3; }

static __device__ __noinline__ void scan_drifting_masked(const uint32_t *row, const uint32_t *__restrict__ mrow, int W, int k, const double *ppm,
                                                  const int *f0, const int *cn, int Mn, double pc, double alpha_pc, int lane,
                                                  double &hv_out, int &w_out) {
    const int B = (W + 31) >> 5;
    const int w_begin = min(W, lane * B), w_end = min(W, w_begin + B);
    // byte-packed occurrences of A,C,G,T in the window (masked bases excluded) + the masked count
    auto add = [&](uint32_t &occ, int &om, int pos, int sign) {
        if (mask_at(mrow, pos)) om += sign;
        else occ += (uint32_t)sign << (8 * base_at(row, pos));
    };
    int blocksum[5] = {0, 0, 0, 0, 0};
    if (w_begin < w_end) {
        uint32_t occ = 0;
        int om = 0;
        for (int j = 0; j < k; ++j) add(occ, om, w_begin + j, 1);
        for (int w = w_begin; w < w_end; ++w) {
#pragma unroll
            for (int b = 0; b < 4; ++b) blocksum[b] += (int)((occ >> (8 * b)) & 255u);
            blocksum[4] += om;
            if (w + 1 < w_end) {
                add(occ, om, w, -1);
                add(occ, om, w + k, 1);
            }
        }
    }
    int run[5];
#pragma unroll
    for (int b = 0; b < 5; ++b) {
        int v = blocksum[b];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, v, o);
            if (lane >= o) v += t;
        }
        run[b] = v - blocksum[b];
    }
    double hv = 0.0;
    int hw = 0;
    if (w_begin < w_end) {
        uint32_t oc = 0;
        int om = 0;
        for (int j = 0; j < k; ++j) add(oc, om, w_begin + j, 1);
        for (int w = w_begin; w < w_end; ++w) {
            int F[4], sum = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                run[b] += (int)((oc >> (8 * b)) & 255u);
                F[b] = f0[b] + (w + 1) * cn[b] - run[b];
                sum += F[b];
            }
            run[4] += om;
            sum += (w + 1) * Mn - run[4];                                         // the dead rows (fs:116 sums every slot)
            if (om == 0) {                                                          // else the window scores 0
                const double den = __dadd_rn((double)sum, alpha_pc);
                double pcv[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) pcv[b] = __ddiv_rn(__dadd_rn((double)F[b], pc), den);
                double v = 1.0;
                for (int j = 0; j < k; ++j) {
                    const int b = base_at(row, w + j);
                    const double q = b == 0 ? pcv[0] : b == 1 ? pcv[1] : b == 2 ? pcv[2] : pcv[3];
                    v = __dmul_rn(v, __ddiv_rn(ppm[j * 4 + b], q));
                }
                if (v > hv) {
                    hv = v;
                    hw = w;
                }
            }
            if (w + 1 < w_end) {
                add(oc, om, w, -1);
                add(oc, om, w + k, 1);
            }
        }
    }
    warp_argmax(hv, hw);
    hv_out = hv;
    w_out = hw;
}

// The same scan when Gap '-' is a member of the alphabet (a.gap_total > 0): Gap is not dead, fuseFrequencyVectors keeps
// its row, so it holds F_w[Gap] = f0g + (w + 1) g_n - sum_{m <= w} gapocc_m like a base (f0g = the others' Gaps outside
// their sites, g_n = the Gaps of this sequence), and a window over a Gap multiplies in P[Gap, j] / q_w[Gap] (gcol[j] =
// P[Gap, j]). Mn counts Gaps too; the dead symbols are Mn - g_n. (A function of its own: sets whose Gap is dead keep
// the scan above as it was.)
static __device__ __noinline__ void scan_drifting_gapped(const uint32_t *row, const uint32_t *__restrict__ mrow, int W, int k, const double *ppm,
                                                  const int *f0, const int *cn, int Mn, double pc, double alpha_pc, int lane,
                                                  double &hv_out, int &w_out, const double *gcol, int f0g, int gn) {
    const int B = (W + 31) >> 5;
    const int w_begin = min(W, lane * B), w_end = min(W, w_begin + B);
    const int Md = Mn - gn; // dead symbols of the sequence
    // byte-packed occurrences of A,C,G,T in the window (masked bases excluded) + the dead count + the Gap count
    auto add = [&](uint32_t &occ, int &om, int &og, int pos, int sign) {
        const int m = mask2_at(mrow, pos);
        if (m == 0) occ += (uint32_t)sign << (8 * base_at(row, pos));
        else if (m == 1) og += sign;
        else om += sign;
    };
    int blocksum[6] = {0, 0, 0, 0, 0, 0};
    if (w_begin < w_end) {
        uint32_t occ = 0;
        int om = 0, og = 0;
        for (int j = 0; j < k; ++j) add(occ, om, og, w_begin + j, 1);
        for (int w = w_begin; w < w_end; ++w) {
#pragma unroll
            for (int b = 0; b < 4; ++b) blocksum[b] += (int)((occ >> (8 * b)) & 255u);
            blocksum[4] += om;
            blocksum[5] += og;
            if (w + 1 < w_end) {
                add(occ, om, og, w, -1);
                add(occ, om, og, w + k, 1);
            }
        }
    }
    int run[6];
#pragma unroll
    for (int b = 0; b < 6; ++b) {
        int v = blocksum[b];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, v, o);
            if (lane >= o) v += t;
        }
        run[b] = v - blocksum[b];
    }
    double hv = 0.0;
    int hw = 0;
    if (w_begin < w_end) {
        uint32_t oc = 0;
        int om = 0, og = 0;
        for (int j = 0; j < k; ++j) add(oc, om, og, w_begin + j, 1);
        for (int w = w_begin; w < w_end; ++w) {
            int F[4], sum = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                run[b] += (int)((oc >> (8 * b)) & 255u);
                F[b] = f0[b] + (w + 1) * cn[b] - run[b];
                sum += F[b];
            }
            run[4] += om;
            run[5] += og;
            sum += (w + 1) * Md - run[4];                                         // the dead rows (fs:116 sums every slot)
            const int Fg = f0g + (w + 1) * gn - run[5];                             // the Gap row
            sum += Fg;
            if (om == 0) {                                                          // else the window scores 0
                const double den = __dadd_rn((double)sum, alpha_pc);
                double pcv[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) pcv[b] = __ddiv_rn(__dadd_rn((double)F[b], pc), den);
                double v = 1.0;
                if (og == 0) {
                    for (int j = 0; j < k; ++j) {
                        const int b = base_at(row, w + j);
                        const double q = b == 0 ? pcv[0] : b == 1 ? pcv[1] : b == 2 ? pcv[2] : pcv[3];
                        v = __dmul_rn(v, __ddiv_rn(ppm[j * 4 + b], q));
                    }
                } else { // a window over Gaps (no dead symbol here: a masked column is a Gap)
                    const double qg = __ddiv_rn(__dadd_rn((double)Fg, pc), den); // fs:119 for the Gap slot
                    for (int j = 0; j < k; ++j) {
                        const int b = base_at(row, w + j);
                        const double q = b == 0 ? pcv[0] : b == 1 ? pcv[1] : b == 2 ? pcv[2] : pcv[3];
                        double r;
                        if (mask_at(mrow, w + j)) r = __ddiv_rn(gcol[j], qg);
                        else r = __ddiv_rn(ppm[j * 4 + b], q);
                        v = __dmul_rn(v, r);
                    }
                }
                if (v > hv) {
                    hv = v;
                    hw = w;
                }
            }
            if (w + 1 < w_end) {
                add(oc, om, og, w, -1);
                add(oc, om, og, w + k, 1);
            }
        }
    }
    warp_argmax(hv, hw);
    hv_out = hv;
    w_out = hw;
}

// Gap as a member of the alphabet (gap_total > 0, MASKED instantiations only; rare path, out of line): the Gap column of
// the PPM, P[Gap, j] = pvals[C[Gap, j]] (normalizePPM, fs:255-261, like the A,C,G,T rows), into gcol when the held-out
// row holds symbols outside A,C,G,T (mrow != null; only its exact scan reads the column). Returns x = f0[Gap] = the set's
// Gaps - this sequence's - the Gaps of the other sites (fs:565-568, fs:67-69), y = this sequence's Gaps (from its mask
// row). gap = the gap row of the counts (site_counts / random_loo_counts_impl); own_mk = mask k-mer of the own site (0:
// none). Scalars only: a ChainArgs reference would make the caller copy its kernel parameters to local memory.
static __device__ __noinline__ int2 drift_gap_tables(const int32_t *gap, uint64_t own_mk, int k, const double *__restrict__ pvals,
                                                     int gap_total, const uint32_t *__restrict__ mrow, int row_words, double *gcol,
                                                     int lane) {
    int s = 0;
    if (lane < k) { // k <= 32
        int c = gap[lane];
        if (((own_mk >> (2 * lane)) & 3u) == 1u) c -= 1;
        s = c;
        if (mrow != nullptr) gcol[lane] = __ldg(pvals + c);
    }
    int g = 0;
    if (mrow != nullptr)
        for (int i = lane; i < row_words; i += 32) { // pairs 0b01: Gap (the row is zero past its end)
            const uint32_t x = __ldg(mrow + i);
            g += __popc(x & ~(x >> 1) & 0x55555555u);
        }
    const int gn = __reduce_add_sync(FULL, g);
    const int f0g = gap_total - gn - __reduce_add_sync(FULL, s);
    __syncwarp();
    return make_int2(f0g, gn);
}

// ------------------------------------------------------------------------------------------------
// one site update with the drifting background, the pieces chain_kernel<.., DRIFT = true> calls
// ------------------------------------------------------------------------------------------------
// PPM of the leave-one-out counts (createPPMOf + normalizePPM, fs:573-575) into W.wcol, the counts themselves into
// W.lgcol; f0 = fused createFCVWithout of the other sequences (fs:565-568: their bases outside their sites),
// cn = base counts of the held-out sequence; the float32 pair table when the ranking pass is allowed.
// counts = W.counts (random starts) or the all-sites total; use_given = the caller-supplied PPM of fs:644-661.
template <int KP>
__device__ __forceinline__ void drift_tables(const WarpTables &W, const int32_t *counts, bool has_own, uint64_t own, int k,
                                             const ChainArgs &a, bool use_given, bool fast, int n, int lane, int (&f0)[4],
                                             int (&cn)[4], uint64_t own_mask = 0) {
    for (int e = lane; e < 4 * k; e += 32) {
        int c = counts[e];
        if (has_own && (int)((own >> (2 * (e >> 2))) & 3u) == (e & 3) && !((own_mask >> (2 * (e >> 2))) & 1u)) c -= 1; // (a masked own base was never counted)
        W.wcol[e] = use_given ? __ldg(a.ppm_given + e) : __ldg(a.pvals + c);
        W.lgcol[e] = c;
    }
    __syncwarp();
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        int s = 0;
        for (int j = lane; j < k; j += 32) s += W.lgcol[j * 4 + b];
        cn[b] = __ldg(a.basecnt + n * 4 + b);
        f0[b] = (a.gcnt[b] - cn[b]) - __reduce_add_sync(FULL, s);
    }
    // (W.counts was consumed above: its space holds the float32 log table)
    if (fast) drift_pair_table<KP>(W.wcol, reinterpret_cast<float *>(W.counts), reinterpret_cast<float *>(W.ptab), k, lane);
}

// getBestPWMSs (fs:462-479) for the staged row; returns true when every window was scored in float64.
// masked_n >= 0: the held-out sequence holds symbols outside A,C,G,T (a.s.mask != null); seq = its index (prefix tables)
// f0g, gn: f0[Gap] and the held-out sequence's Gaps (drift_gap_tables) when Gap is a member of the alphabet, else 0;
// the Gap column of the PPM is in W.ptab (as float64) for a masked row, which builds no pair table.
template <int KP>
__device__ __forceinline__ bool drift_pick(const WarpTables &W, const uint32_t *row, int Wn, int k, const ChainArgs &a, bool fast,
                                           const int (&f0)[4], const int (&cn)[4], int lane, double &p, int &w, int masked_n = -1,
                                           int seq = -1, int f0g = 0, int gn = 0) {
    if (masked_n >= 0) {
        const uint32_t *mrow = a.s.mask + (size_t)masked_n * a.s.row_words;
        if (a.gap_total > 0)
            scan_drifting_gapped(row, mrow, Wn, k, W.wcol, f0, cn, __ldg(a.maskcnt + masked_n), a.pc, a.alpha_pc, lane, p, w,
                                 reinterpret_cast<const double *>(W.ptab), f0g, gn);
        else
            scan_drifting_masked(row, mrow, Wn, k, W.wcol, f0, cn, __ldg(a.maskcnt + masked_n), a.pc, a.alpha_pc, lane, p, w);
        return true;
    }
    bool ranked = false;
    if (fast && a.ss != nullptr && seq >= 0)
        ranked = scan_drifting_tables<KP>(row, reinterpret_cast<const int4 *>(a.ss) + (size_t)seq * a.ss_stride, Wn, k, W.wcol,
                                          reinterpret_cast<const float *>(W.ptab), f0, cn, f0g, a.pc, a.alpha_pc, lane, p, w);
    else if (fast)
        ranked = scan_drifting_fast<KP>(row, Wn, k, W.wcol, reinterpret_cast<const float *>(W.ptab), f0, cn, f0g, a.pc, a.alpha_pc,
                                        lane, p, w);
    if (!ranked) scan_drifting(row, Wn, k, W.wcol, f0, cn, f0g, a.pc, a.alpha_pc, lane, p, w);
    return !ranked;
}

} // namespace gibbs
