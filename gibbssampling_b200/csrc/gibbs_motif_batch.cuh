// gibbssampling_b200/csrc/gibbs_motif_batch.cuh -- the MotifSampler restarts of many independent sequence sets in one
// launch (gibbs_batch_run_motif_device, include/gibbs_b200.h).
//
// Same layout as chain_batch_kernel (gibbs_batch.cuh): every set has its own Motif2Args in a device array -- its rows, W or
// PPM-value tables, background-only window tables, result slices, roulette error flag and its slices of the scratch lists
// -- and a launch covers one group of sets. CTA g runs restart g - chain_off[j] of set set_ids[j]: thread 0 finds j by
// binary search, copies that set's arguments to shared memory and takes the run-wide fields from the kernel's own
// argument; the restart is then the body of motif_kernel (gibbs_motif_body.inc) or of motif2_kernel
// (gibbs_motif2_body.inc), reading the shared copy. Batches run without the straggler hand-over, and the random starts
// ran before in the batch random-start units (chain_batch_kernel<.., INIT_ONLY>), so run.init_done = 1.
// A set's scratch slice holds R x T lists of its own window stride, indexed by the restart within the set.
#pragma once
#include "gibbs_motif2.cuh"

namespace gibbs {

struct MotifBatchTable {
    const Motif2Args *sets;   // [all sets] per-set arguments (motifAmount = 1 reads .m)
    const int32_t *set_ids;   // [n] the sets of this group
    const int32_t *chain_off; // [n + 1] first restart of each of them in the launch's grid
    int32_t n;
};

// entry of the group that CTA g belongs to: the last j with chain_off[j] <= g
__device__ __forceinline__ int motif_batch_entry(const MotifBatchTable &bt, int g) {
    int lo = 0, hi = bt.n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(bt.chain_off + mid) <= g) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// the run-wide fields of a batch run over a set's own; no hand-over
__device__ __forceinline__ void motif_batch_run_fields(MotifArgs &d, const MotifArgs &run) {
    d.c.seed = run.c.seed;
    d.c.chain_id_base = run.c.chain_id_base; // restart r of every set draws from (seed, chain_id_base + r)
    d.c.rng_mode = run.c.rng_mode;
    d.c.phase_mask = run.c.phase_mask;
    d.c.cutoff = run.c.cutoff;
    d.c.max_sweeps = run.c.max_sweeps;
    d.c.stats = run.c.stats;
    d.c.active = nullptr;
    d.c.pause_below = 0;
    d.c.from_list = 0;
    d.init_done = run.init_done;
}

// Launch bounds, chosen from -Xptxas -v (the body reads its arguments from shared memory, not from the constant bank,
// which costs registers): see DESIGN.md section 4, "Batches".
#ifndef GIBBS_MOTIF_BATCH_T4_BLOCKS
#define GIBBS_MOTIF_BATCH_T4_BLOCKS 5
#endif

template <int KP, int T, bool MASKED>
static __global__ void __launch_bounds__(32 * T, (T == 1 ? 8 : GIBBS_MOTIF_BATCH_T4_BLOCKS)) motif_batch_kernel(const MotifArgs run,
                                                                                                                const MotifBatchTable bt) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int THREADS = 32 * T;
    constexpr int R = (2 * T < 4) ? 4 : 2 * T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ MotifArgs sm;
    __shared__ int32_t s_chain;
    if (tid == 0) {
        const int j = motif_batch_entry(bt, blockIdx.x);
        sm = bt.sets[__ldg(bt.set_ids + j)].m;
        motif_batch_run_fields(sm, run);
        s_chain = blockIdx.x - __ldg(bt.chain_off + j);
    }
    __syncthreads();
    const MotifArgs &m = sm;
    const ChainArgs &a = m.c;
    const int chain = s_chain;
    const TeamSmem S = carve_smem(smem_raw, T);
    const WarpTables WT = warp_tables(S, warp);
    require_aligned_tables(WT);
    int32_t *bsum = reinterpret_cast<int32_t *>(smem_raw + MOTIF_BSUM_OFFSET); // data background: base counts over the sequences that have a site
    const int N = a.s.n, k = a.k;
    int32_t *sites = a.sites + (size_t)chain * N;
    double *pw = a.scores + (size_t)chain * N; // PWMS of the MotifIndex state
    double *hv = a.hv + (size_t)chain * N;
    double *cand_l = m.cand_l + ((size_t)chain * T + warp) * m.bg.wstride;
    int32_t *cand_w = m.cand_w + ((size_t)chain * T + warp) * m.bg.wstride;
    double *gbuf = m.data_bg ? m.gbuf + ((size_t)chain * T + warp) * m.bg.wstride : nullptr;
#include "gibbs_motif_body.inc"
}

template <int KP>
static __global__ void __launch_bounds__(32) motif2_batch_kernel(const MotifArgs run, const MotifBatchTable bt) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    __shared__ Motif2Args sq;
    __shared__ int32_t s_chain;
    if (lane == 0) {
        const int j = motif_batch_entry(bt, blockIdx.x);
        sq = bt.sets[__ldg(bt.set_ids + j)];
        motif_batch_run_fields(sq.m, run);
        s_chain = blockIdx.x - __ldg(bt.chain_off + j);
    }
    __syncthreads();
    const MotifArgs &m = sq.m;
    const ChainArgs &a = m.c;
    const int chain = s_chain;
    const TeamSmem S = carve_smem(smem_raw, 1);
    const WarpTables WT = warp_tables(S, 0);
    require_aligned_tables(WT);
    const int N = a.s.n, k = a.k;
    int32_t *pos2 = sq.pos2 + (size_t)chain * N * 2;
    int32_t *sites = a.sites + (size_t)chain * N; // newest position of every sequence (what the m = 1 calls return)
    double *pw = a.scores + (size_t)chain * N;
    double *hv = a.hv + (size_t)chain * N;
    double *cand_l = m.cand_l + (size_t)chain * m.bg.wstride;
    int32_t *cand_w = m.cand_w + (size_t)chain * m.bg.wstride;
    double *gbuf = m.data_bg ? m.gbuf + (size_t)chain * m.bg.wstride : nullptr;
    double *sc = sq.sc + (size_t)chain * m.bg.wstride;
#include "gibbs_motif2_body.inc"
}

} // namespace gibbs
