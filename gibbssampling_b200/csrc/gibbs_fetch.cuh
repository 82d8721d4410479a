// gibbssampling_b200/csrc/gibbs_fetch.cuh -- the kernels of the winner fetches (gibbs_fetch_best, gibbs_batch_fetch_best,
// gibbs_fetch with counts): the promote-or-restart loop of a run and the PWM counts of its winners.
// Only gibbs_api.cu includes this header. Every kernel unit compiles the static kernels of the headers it includes,
// launched or not, so keeping these out of gibbs_kernels.cuh and gibbs_batch.cuh keeps them out of the kernel units.
#pragma once
#include "gibbs_kernels.cuh"

namespace gibbs {

// counts of all N sites of one chain (PWM counts reported with the best chain)
template <int KP>
static __global__ void __launch_bounds__(32) all_counts_kernel(DeviceSeqs s, const int32_t *sites, int k, int32_t *counts_out) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    const TeamSmem S = carve_smem(smem_raw, 1);
    if (lane < 16) S.lut[lane] = hist_lut_entry(lane);
    __syncwarp();
    site_counts<KP, 1>(s, sites, -1, k, SHIFT_NONE, S.total, S.lut, S.fix, lane);
    for (int e = lane; e < k * 4; e += 32) counts_out[e] = S.total[e];
}

// all_counts_kernel once per set: PWM counts [set][k][4] of the winners' sites (-1 = none: all zero)
template <int KP>
static __global__ void __launch_bounds__(32) all_counts_batch_kernel(const ChainArgs *sets, const int32_t *seq_off, const int32_t *sites,
                                                                     int k, int32_t *counts_out) {
    __shared__ int32_t total[MAX_COLS * 4];
    __shared__ uint32_t lut[16];
    __shared__ int32_t fix[MAX_COLS];
    const int s = blockIdx.x, lane = threadIdx.x;
    if (lane < 16) lut[lane] = hist_lut_entry(lane);
    __syncwarp();
    const DeviceSeqs ds = sets[s].s;
    site_counts<KP, 1>(ds, sites + seq_off[s], -1, k, SHIFT_NONE, total, lut, fix, lane);
    for (int e = lane; e < k * 4; e += 32) counts_out[(size_t)s * k * 4 + e] = total[e];
}

// ------------------------------------------------------------------------------------------------
// the promote-or-restart loop of fs:435-459 (= fs:616-640, fs:665-689, fs:857-881, fs:974-998; quirk A.6-8), decided on
// the device over the restarts of one run (chain r = restart r)
// ------------------------------------------------------------------------------------------------
//   loop n acc best:  n > reps -> best | acc = best -> best | sum acc > sum best -> loop (n+1) [||] (acc unless empty)
//                     | else -> loop (n+1) (next restart) best          starting from  loop 0 [||] [|(0., 0)|]
// Every restart costs one iteration and every promotion one more, so restart r sits in `acc` at iteration
// r + 1 + 2 * (promotions so far). One warp walks the sums 32 restarts at a time and stops only at EVENTS: the iteration
// cap, a sum equal to the best one (acc = best needs the arrays compared, rare) or a larger sum (promotion). A promoted
// restart with a negative sum ends the loop (0. > sum best then burns the remaining iterations without running anything).
// out[0] = index of the returned restart, -1 = the initial value survived (the caller returns [|(0., 0)|]);
// the winner's rows are copied to win_sites / win_scores so that one fixed-address copy brings them to the host.
// motif = the MotifIndex flavour of the initial value: {PWMS 0.; Positions []} (site -1) instead of (0., 0).
// NS = site entries per restart: N, or 2 N for Positions lists of up to two sites (motifAmount = 2).
static __global__ void __launch_bounds__(32) restart_select_kernel(const double *sums, const int32_t *sites, const double *scores,
                                                                   int n_chains, int N, int NS, int reps, int motif, int32_t *out,
                                                                   int32_t *win_sites, double *win_scores, double *win_sum) {
    const int lane = threadIdx.x;
#include "gibbs_restart_select_body.inc" // (shared with restart_select_batch_kernel)
}

// restart_select_kernel once per set (one warp each), for either sampler: sums [set][R], scores [set][R][N_s] at
// R seq_off[set], sites [set][R][N_s][m] at m R seq_off[set] (m = 2: the Positions lists); winners' sites at m seq_off[set]
static __global__ void __launch_bounds__(32) restart_select_batch_kernel(const double *all_sums, const int32_t *all_sites,
                                                                         const double *all_scores, const int32_t *seq_off, int n_chains,
                                                                         int reps, int m, int motif, int32_t *best_out,
                                                                         int32_t *all_win_sites, double *all_win_scores, double *win_sums) {
    const int set = blockIdx.x, lane = threadIdx.x;
    const int o = seq_off[set], N = seq_off[set + 1] - o, NS = m * N;
    const size_t cells = (size_t)n_chains * o;
    const double *sums = all_sums + (size_t)set * n_chains;
    const int32_t *sites = all_sites + cells * m;
    const double *scores = all_scores + cells;
    int32_t *out = best_out + set, *win_sites = all_win_sites + (size_t)m * o;
    double *win_scores = all_win_scores + o, *win_sum = win_sums + set;
#include "gibbs_restart_select_body.inc"
}

// element `which` of every Positions pair: the site arrays the one-site kernels take
static __global__ void pair_element_kernel(const int32_t *pos2, int n, int which, int32_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = pos2[2 * i + which];
}

} // namespace gibbs
