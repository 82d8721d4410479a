// gibbssampling_b200/csrc/gibbs_batch.cuh -- many independent sequence sets in one launch (gibbs_batch_*, include/gibbs_b200.h).
//
// A batch is S sets uploaded as one concatenation (common row_words). Every set has its own ChainArgs -- its rows, W table,
// drift tables and result slices -- in a device array; a launch covers one GROUP of sets that share a team size and the
// masked flag. CTA g of a launch runs chain g - chain_off[j] of set set_ids[j], j = the last entry with chain_off[j] <= g:
// thread 0 finds j by binary search, copies that set's ChainArgs to shared memory and takes the run-wide fields from the
// kernel's own argument; the restart is then the body of chain_kernel (gibbs_chain_body.inc), reading the shared copy.
// Batches run without the straggler hand-over.
#pragma once
#include "gibbs_kernels.cuh"

namespace gibbs {

struct BatchTable {
    const ChainArgs *sets;    // [all sets] per-set arguments (rows, tables, result slices)
    const int32_t *set_ids;   // [n] the sets of this group
    const int32_t *chain_off; // [n + 1] first chain of each of them in the launch's grid
    int32_t n;
};

// Launch bounds of the batch instantiations, chosen from -Xptxas -v (not those of chain_kernel: the body reads its
// arguments from shared memory, not from the constant bank, which costs registers). 4-warp sweeps: 6 CTAs per SM
// (80 registers; at chain_kernel's 7 / 72 registers 9 of 16 k-widths spilled), with the drifting background 5 CTAs
// (96 registers; at 80 every k-width spilled, up to 120 B of stores).
#ifndef GIBBS_BATCH_T4_MIN_BLOCKS
#define GIBBS_BATCH_T4_MIN_BLOCKS 6
#endif
#ifndef GIBBS_BATCH_T4_DRIFT_MIN_BLOCKS
#define GIBBS_BATCH_T4_DRIFT_MIN_BLOCKS 5
#endif
#define GIBBS_BATCH_MIN_BLOCKS(T, DRIFT, INIT_ONLY) \
    (INIT_ONLY ? (T == 1 ? 8 : 4) : T == 1 ? 16 : DRIFT ? GIBBS_BATCH_T4_DRIFT_MIN_BLOCKS : GIBBS_BATCH_T4_MIN_BLOCKS)

template <int KP, int T, bool MASKED, bool DRIFT, bool INIT_ONLY>
static __global__ void __launch_bounds__(32 * T, GIBBS_BATCH_MIN_BLOCKS(T, DRIFT, INIT_ONLY)) chain_batch_kernel(const ChainArgs run, const BatchTable bt) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int THREADS = 32 * T;
    constexpr int R = (2 * T < 4) ? 4 : 2 * T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ ChainArgs sa;
    __shared__ int32_t s_chain;
    if (tid == 0) {
        const int g = blockIdx.x;
        int lo = 0, hi = bt.n - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (__ldg(bt.chain_off + mid) <= g) lo = mid;
            else hi = mid - 1;
        }
        sa = bt.sets[__ldg(bt.set_ids + lo)];
        sa.seed = run.seed;
        sa.chain_id_base = run.chain_id_base; // restart r of every set draws from (seed, chain_id_base + r)
        sa.rng_mode = run.rng_mode;
        sa.phase_mask = run.phase_mask;
        sa.max_sweeps = run.max_sweeps;
        sa.min_width = run.min_width;
        sa.stats = run.stats;
        sa.active = nullptr;
        sa.pause_below = 0;
        sa.from_list = 0;
        s_chain = g - __ldg(bt.chain_off + lo);
    }
    __syncthreads();
    const ChainArgs &a = sa;
    const int chain = s_chain;
#include "gibbs_chain_body.inc"
}

} // namespace gibbs
