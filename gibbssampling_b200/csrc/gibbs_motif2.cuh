// gibbssampling_b200/csrc/gibbs_motif2.cuh -- MotifSampler with motifAmount = 2 (fs:727-742 driven by fs:778-782; the
// reference script's second live call, fsx:407): up to two non-overlapping sites per sequence.
//
// The candidate list of one held-out sequence is (fs:759-784)
//     [W background entries] ++ [single windows with log2 score > cutOff] ++ [pairs i < j, more than k apart,
//                                                                            log2(score_i) > cutOff and log2(score_j score_i) > cutOff]
// in that order: calculatePWMsForSegmentCombinations walks the windows include-first, so pairs come in
// lexicographic order, and a pair's PWMS is log2 of the float64 product score_j * (score_i * 1.0), its Positions [j; i]
// (newest first, fs:736). The list is never materialised: every window's float64 product is written once, the single
// candidates are compacted, and the pairs are streamed 32 at a time in list order -- twice for the roulette (List.sum,
// then the walk of fs:746-754, both in the reference's sequential float64 order) and once for the greedy head (first
// maximum by PWMS = head of the stable List.sortByDescending, fs:812 / fs:919).
// One warp runs one chain (= one restart): this family trades the team machinery of motif_kernel for exactness and
// reviewability; the number of pairs grows with the square of the candidates, so it is not a throughput path.
#pragma once
#include "gibbs_motif.cuh"

namespace gibbs {

struct Motif2Args {
    MotifArgs m;       // tables, scratch and flags of the m = 1 family (cand_l / cand_w / gbuf: one list per chain)
    int32_t *pos2;     // [chains][n][2] Positions of every sequence, newest first (fs:736); -1 = absent
    double *sc;        // [chains][wstride] float64 window products of the current held-out sequence
};

// sequential float64 accumulation over a stream of list items handed over 32 at a time (lane order = list order)
struct ListWalk {
    double sum;   // List.sum of all PWMS (fs:748)
    double acc;   // running lower bound of the walk (fs:750-753)
    double pick;
    int found;    // 0 / 1
    double sel_v; // PWMS of the selected item
    int sel_a, sel_b; // its positions: (-1, -1) background, (w, -1) single, (j, i) pair
};

// pass 1: sum += v over the valid lanes, in lane order
__device__ __forceinline__ void list_sum_block(ListWalk &L, double v, bool valid) {
    unsigned m = __ballot_sync(FULL, valid);
    while (m) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        L.sum = __dadd_rn(L.sum, __shfl_sync(FULL, v, j));
    }
}
// pass 2: the walk; a, b = positions of this lane's item
__device__ __forceinline__ void list_walk_block(ListWalk &L, double v, bool valid, int a, int b) {
    if (L.found) return;
    const double wgt = __ddiv_rn(v, L.sum); // divisions in parallel, accumulation in list order
    unsigned m = __ballot_sync(FULL, valid);
    while (m) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        const double hi = __dadd_rn(L.acc, __shfl_sync(FULL, wgt, j));
        if (L.acc <= L.pick && L.pick <= hi) {
            L.found = 1;
            L.sel_v = __shfl_sync(FULL, v, j);
            L.sel_a = __shfl_sync(FULL, a, j);
            L.sel_b = __shfl_sync(FULL, b, j);
            return;
        }
        L.acc = hi;
    }
}

// first maximum in list order over a stream: (value, order key) with the smaller key winning ties
struct ListHead {
    double v;
    long long key;
    int a, b;
};
__device__ __forceinline__ void head_offer(ListHead &H, double v, long long key, int a, int b) {
    if (v > H.v || (v == H.v && key < H.key)) {
        H.v = v;
        H.key = key;
        H.a = a;
        H.b = b;
    }
}
__device__ __forceinline__ void head_reduce(ListHead &H) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double ov = __shfl_xor_sync(FULL, H.v, o);
        const long long ok = __shfl_xor_sync(FULL, H.key, o);
        const int oa = __shfl_xor_sync(FULL, H.a, o), ob = __shfl_xor_sync(FULL, H.b, o);
        if (ov > H.v || (ov == H.v && ok < H.key)) {
            H.v = ov;
            H.key = ok;
            H.a = oa;
            H.b = ob;
        }
    }
}

// pairs (i, j) of the list, streamed in list order. F(l, valid, j, i, order key) is called once per block of 32
// second windows, by the whole warp.
template <typename F>
__device__ __forceinline__ void for_each_pair_block(const double *sc, const int32_t *cand_w, int n_single, int W, int k,
                                                    double cutoff, int lane, F &&f) {
    for (int ci = 0; ci < n_single; ++ci) {
        const int wi = cand_w[ci];
        const double pi = __dmul_rn(sc[wi], 1.0); // fs:735: scores.[n] * prob with prob = 1.
        for (int j0 = wi + k + 1; j0 < W; j0 += 32) { // fs:129-140: |j - i| > motifLength
            const int j = j0 + lane;
            double l = 0.0;
            bool valid = false;
            if (j < W) {
                l = log2_ref(__dmul_rn(sc[j], pi));
                valid = l > cutoff;
            }
            f(l, valid, j, wi, (long long)ci * W + j);
        }
    }
}

template <int KP>
static __global__ void __launch_bounds__(32) motif2_kernel(const Motif2Args q) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const MotifArgs &m = q.m;
    const ChainArgs &a = m.c;
    const int lane = threadIdx.x;
    const int chain = blockIdx.x;
    const TeamSmem S = carve_smem(smem_raw, 1);
    const WarpTables WT = warp_tables(S, 0);
    require_aligned_tables(WT);
    const int N = a.s.n, k = a.k;
    int32_t *pos2 = q.pos2 + (size_t)chain * N * 2;
    int32_t *sites = a.sites + (size_t)chain * N; // newest position of every sequence (what the m = 1 calls return)
    double *pw = a.scores + (size_t)chain * N;
    double *hv = a.hv + (size_t)chain * N;
    double *cand_l = m.cand_l + (size_t)chain * m.bg.wstride;
    int32_t *cand_w = m.cand_w + (size_t)chain * m.bg.wstride;
    double *gbuf = m.data_bg ? m.gbuf + (size_t)chain * m.bg.wstride : nullptr;
    double *sc = q.sc + (size_t)chain * m.bg.wstride;
#include "gibbs_motif2_body.inc"
}

// start state of a run without the random starts: Positions lists from the one-site state of gibbs_set_start_state
static __global__ void motif2_seed_kernel(const int32_t *sites, long long cells, int32_t *pos2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cells) {
        pos2[2 * i] = sites[i];
        pos2[2 * i + 1] = -1;
    }
}

} // namespace gibbs
