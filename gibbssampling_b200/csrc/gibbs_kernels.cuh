// gibbssampling_b200/csrc/gibbs_kernels.cuh -- __global__ kernels (sm_100a only).
#pragma once
#include "gibbs_device.cuh"
#include "gibbs_drift_dev.cuh"

namespace gibbs {

enum Phase { PH_INIT = 0, PH_GREEDY = 1, PH_LEFT = 2, PH_RIGHT = 3, PH_DONE = 4 };

// first phase >= from whose bit (1 << phase) is set in mask
__device__ __forceinline__ int next_phase(int from, int mask) {
    int ph = from;
    while (ph < PH_DONE && !((mask >> ph) & 1)) ++ph;
    return ph;
}

// ------------------------------------------------------------------------------------------------
// setup kernels
// ------------------------------------------------------------------------------------------------
// ASCII -> 2-bit rows + mask plane. One thread per packed word.
// flags[0] = 1 + a byte outside '*'..'Z' (the reference's 49-slot tables cannot index it: IndexOutOfRange, fs:17-20)
// flags[1] = number of symbols inside that range but outside A,C,G,T (mask plane 0b11, code 0)
// flags[2] = 1 if one of them is Gap '-' (a member of the script's alphabet, fsx:368-369)
static __global__ void pack_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off, int n, int row_words,
                            uint32_t *__restrict__ packed, uint32_t *__restrict__ mask, int32_t *__restrict__ rowflag,
                            int32_t *__restrict__ len_out, int *flags) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)n * row_words) return;
    const int i = (int)(t / row_words), wd = (int)(t % row_words);
    const int64_t o = off[i];
    const int len = (int)(off[i + 1] - o);
    if (wd == 0) len_out[i] = len;
    uint32_t v = 0, m = 0;
    int other = 0;
    const int b0 = wd * 16;
#pragma unroll
    for (int x = 0; x < 16; ++x) {
        const int b = b0 + x;
        if (b < len) {
            const uint8_t c = ascii[o + b];
            uint32_t code = 0;
            if (c == 'A') code = 0;
            else if (c == 'C') code = 1;
            else if (c == 'G') code = 2;
            else if (c == 'T') code = 3;
            else if (c >= 42 && c <= 90) {
                m |= 3u << (2 * x);
                ++other;
                if (c == '-') atomicExch(flags + 2, 1);
            } else {
                atomicExch(flags, 1 + (int)c);
            }
            v |= code << (2 * x);
        }
    }
    packed[t] = v;
    mask[t] = m;
    if (other) {
        atomicAdd(flags + 1, other);
        rowflag[i] = 1;
    }
}

// gather copy of the packed rows: wide[i][m] = 64 bits from bit 16 m of row i (see DeviceSeqs::wide). One thread per word.
static __global__ void wide_kernel(const uint32_t *__restrict__ packed, int n, int row_words, int wide_words, uint64_t *__restrict__ wide) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)n * wide_words) return;
    const int i = (int)(t / wide_words), m = (int)(t % wide_words);
    const uint32_t *row = packed + (size_t)i * row_words;
    const int w = m >> 1; // 16 m bits = word m / 2 (+ 16 bits for odd m); rows end in >= 4 zero words
    uint32_t a = row[w], b = w + 1 < row_words ? row[w + 1] : 0u, c = w + 2 < row_words ? row[w + 2] : 0u;
    uint64_t v = ((uint64_t)b << 32) | a;
    if (m & 1) v = (v >> 16) | ((uint64_t)c << 48);
    wide[t] = v;
}

// W(c, b) = ((c + pc) / den) / q[b]   (normalizePPM fs:260, createPositionWeightMatrix fs:286)
// plus its fixed-point log2. range[0] = min lg, range[1] = max lg, range[2] = any non-normal W.
static __global__ void wtab_kernel(int n, double pc, double den, double q0, double q1, double q2, double q3, WEnt *wtab,
                            int *range) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * 4) return;
    const int c = t >> 2, b = t & 3;
    const double q = b == 0 ? q0 : b == 1 ? q1 : b == 2 ? q2 : q3;
    const double w = __ddiv_rn(__ddiv_rn(__dadd_rn((double)c, pc), den), q);
    WEnt e;
    e.w = w;
    e.pad = 0;
    const bool normal = (w >= 2.2250738585072014e-308) && (w <= 1.7976931348623157e308);
    if (normal) {
        double units = rint(log2(w) * (double)(1 << LG_FRAC_BITS));
        units = fmin(fmax(units, -4000000.0), 4000000.0);
        const int u = (int)units;
        e.lg = u * (1 << KEY_IDX_BITS);
        atomicMin(&range[0], u);
        atomicMax(&range[1], u);
    } else {
        e.lg = 0;
        atomicExch(&range[2], 1);
    }
    wtab[t] = e;
}

// ------------------------------------------------------------------------------------------------
// uniform stream -> leave-one-out counts of the random initial sites (fs:418-426), one warp
// ------------------------------------------------------------------------------------------------
// Draw index of (held-out n, other sequence i) = n (N-1) + rank of i among the others, the order in
// which the reference's Array.map consumes System.Random (fs:419-421, quirk A.6-5). Each lane
// takes one Philox block (4 draws) per round; the 4 draws are processed branch-free so their
// length / row loads overlap.
// NB = Philox blocks per lane per round: 4 NB independent gathers in flight per lane.
#ifndef GIBBS_P0_NB_CHAIN
#define GIBBS_P0_NB_CHAIN 1
#endif
#ifndef GIBBS_P0_NB_INIT_SMALL
#define GIBBS_P0_NB_INIT_SMALL 4
#endif
#ifndef GIBBS_P0_NB_INIT_LARGE
#define GIBBS_P0_NB_INIT_LARGE 2
#endif
#ifndef GIBBS_T4_MIN_BLOCKS
#define GIBBS_T4_MIN_BLOCKS 7 // 72 registers per thread; measured against 6 (80) and 8 (64)
#endif
#ifndef GIBBS_T8_MIN_BLOCKS
#define GIBBS_T8_MIN_BLOCKS 3
#endif
#ifndef GIBBS_T16_MIN_BLOCKS
#define GIBBS_T16_MIN_BLOCKS 1
#endif
#ifndef GIBBS_INIT_MIN_BLOCKS
#define GIBBS_INIT_MIN_BLOCKS 2
#endif
// MASKED = the set holds symbols outside A,C,G,T: a separate instantiation, so that the ACGT loop stays free of calls
// and keeps its loads batched (with the check inline the random starts of C2 cost 60 % more instructions).
// SROWS = `rows` is a copy of the packed set in shared memory (init_smem_kernel): the gathers are LDS, not L1 sectors.
// The base counts are kept bit-sliced in registers (KmerCounter): no lookup table.
// UNI = every sequence has the same length (no length load per draw); PHILOX = the counter-based stream (else the
// injected doubles): warp-uniform properties of the run, hoisted out of the draw loop as template parameters.
// WIDE = gather from the 64-bit copy (DeviceSeqs::wide) instead of the packed rows in global memory.
template <int KP, int NB, bool MASKED, bool SROWS, bool UNI, bool PHILOX, bool WIDE = false>
__device__ __forceinline__ void random_draw_loop(const ChainArgs &a, uint64_t chain_uid, int chain_local, int n, int32_t *counts,
                                                 int lane, int32_t *fix, const uint32_t *base_rows) {
    using Word = typename KmerCounter<KP>::Word;
    const int N = a.s.n, k = a.k;
    const int row_words = a.s.row_words;
    const uint64_t base = (uint64_t)n * (uint64_t)(N - 1);
    const uint64_t d_end = base + (uint64_t)(N - 1);
    const uint64_t blk0 = base >> 2, blk1 = (d_end + 3) >> 2;
    const int n_blk = (int)(blk1 - blk0);
    const int iters = (n_blk + 32 * NB - 1) / (32 * NB);
    const int r_first = (int)((int64_t)(blk0 << 2) - (int64_t)base); // rank of the first draw of block blk0: -3 .. 0
    const uint32_t range_u = (uint32_t)(a.s.uniform_len - k + 1);
    KmerCounter<KP> h;
    h.clear();
    constexpr int FLUSH_ROUNDS = 63 / NB; // 63 quads = 252 k-mers per lane between warp reductions
    bool first = true;
    for (int it0 = 0; it0 < iters; it0 += FLUSH_ROUNDS) {
        const int it1 = min(iters, it0 + FLUSH_ROUNDS);
        for (int it = it0; it < it1; ++it) {
            Word kmer[NB][4];
#pragma unroll
            for (int q = 0; q < NB; ++q) {
                const int bi = (it * NB + q) * 32 + lane; // block index inside this held-out sequence's draw range
                uint32_t wd[4] = {0, 0, 0, 0};
                if (PHILOX) {
                    const uint64_t blk = blk0 + (uint64_t)bi;
                    const uint4 r = philox4x32_10(make_uint4((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)chain_uid, (uint32_t)(chain_uid >> 32)),
                                                  make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
                    wd[0] = r.x; wd[1] = r.y; wd[2] = r.z; wd[3] = r.w;
                }
                const int r0 = r_first + 4 * bi; // rank of draw 0 of this block; a draw is valid iff 0 <= rank < N-1
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const bool ok = (unsigned)(r0 + x) < (unsigned)(N - 1);
                    const int r = ok ? r0 + x : 0;
                    const int i = r + (r >= n ? 1 : 0); // always a valid sequence index (N >= 2)
                    const uint32_t range = UNI ? range_u : (uint32_t)(__ldg(a.s.len + i) - k + 1);
                    int pos;
                    if (PHILOX) {
                        pos = (int)__umulhi(wd[x], range); // floor(word * 2^-32 * range), exact
                    } else {
                        const int64_t d = (int64_t)base + r;
                        const double u = d < a.uniforms_per_chain ? __ldg(a.uniforms + (size_t)chain_local * a.uniforms_per_chain + d)
                                                                  : 0.0; // (the host rejects streams that are too short)
                        pos = (int)(u * (double)range);           // rnd.Next(0, L-k+1), fs:145
                        pos = min(max(pos, 0), (int)range - 1);   // memory safety for u outside [0,1)
                    }
                    const Word km = WIDE ? gather_kmer_wide<KP>(a.s.wide, a.s.wide_words, i, pos) : gather_kmer<KP, SROWS>(base_rows, row_words, i, pos);
                    kmer[q][x] = ok ? km : (Word)0; // code 0 in every column: counted nowhere
                    if (MASKED && ok && __ldg(a.s.rowflag + i) != 0) hist_fix(a.s.mask, row_words, i, pos, k, fix);
                }
            }
#pragma unroll
            for (int q = 0; q < NB; ++q) h.add4(kmer[q]);
        }
        h.flush(counts, k, it1 == iters ? N - 1 : 0, first, lane);
        first = false;
    }
    KmerCounter<KP>::finish(counts, k, lane);
}

template <int KP, int NB, bool MASKED, bool SROWS = false>
__device__ __forceinline__ void random_loo_counts_impl(const ChainArgs &a, uint64_t chain_uid, int chain_local, int n,
                                                       int32_t *counts, int lane, int32_t *fix,
                                                       const uint32_t *rows = nullptr) {
    const int N = a.s.n, k = a.k;
    if (MASKED) fix[lane] = 0; // fix[] = the warp's lgcol, free until build_tables
    if (N < 2) {
        for (int e = lane; e < 8 * KP; e += 32) counts[e] = 0;
        __syncwarp();
        return;
    }
    const uint32_t *const base_rows = SROWS ? rows : a.s.packed;
    bool done = false;
    if constexpr (!SROWS && KP <= 13) { // the 64-bit gather copy holds every k-mer of k <= 25 in one aligned word
        if (a.rng_mode == 0 && a.s.wide != nullptr && k <= 25) {
            if (a.s.uniform_len > 0) random_draw_loop<KP, NB, MASKED, false, true, true, true>(a, chain_uid, chain_local, n, counts, lane, fix, base_rows);
            else random_draw_loop<KP, NB, MASKED, false, false, true, true>(a, chain_uid, chain_local, n, counts, lane, fix, base_rows);
            done = true;
        }
    }
    if (done) {
    } else if (a.rng_mode != 0) random_draw_loop<KP, 1, MASKED, SROWS, false, false>(a, chain_uid, chain_local, n, counts, lane, fix, base_rows);
    else if (a.s.uniform_len > 0) random_draw_loop<KP, NB, MASKED, SROWS, true, true>(a, chain_uid, chain_local, n, counts, lane, fix, base_rows);
    else random_draw_loop<KP, NB, MASKED, SROWS, false, true>(a, chain_uid, chain_local, n, counts, lane, fix, base_rows);
    if (MASKED) {
        if (lane < k) counts[lane * 4] -= fix[lane];
        __syncwarp();
    }
}

// The same routine out of line, for kernels whose register budget belongs to their sweeps (chain_kernel sits at 72
// registers; its INIT phase runs once per restart, and at the benchmarked shapes a grid-wide kernel runs it instead).
template <int KP, bool MASKED>
static __device__ __noinline__ void random_loo_counts_call(const ChainArgs &a, uint64_t chain_uid, int chain_local, int n,
                                                           int32_t *counts, int lane, int32_t *fix) {
    random_loo_counts_impl<KP, GIBBS_P0_NB_CHAIN, MASKED>(a, chain_uid, chain_local, n, counts, lane, fix);
}

// ------------------------------------------------------------------------------------------------
// random starts (fs:412-430) as a grid-wide kernel
// ------------------------------------------------------------------------------------------------
// Every (chain, held-out sequence) pair of the random-start sweep is an independent site update (each
// draws fresh sites for all the other sequences), so the sweep is spread over the whole GPU instead of
// over the few warps of the chain's own team: one warp per work item, grid-stride over chains x N items,
// each warp staging its rows through a private two-slot TMA pipeline. This is what keeps the N(N-1)
// draws per restart of large sets (C4: 1e10 per chain) from running on a handful of warps.
constexpr int INIT_WARPS = 8;

__host__ __device__ inline int init_smem_bytes(int row_words) {
    return 64 + INIT_WARPS * 16 + INIT_WARPS * WARP_TABLE_BYTES + INIT_WARPS * 2 * row_words * 4;
}

// DRIFT = the data-derived background (getPWMOfRandomStarts fs:589-611, getMotifsWithBestPWMSOfPPM fs:644-661)
template <int KP, bool DRIFT = false>
static __global__ void __launch_bounds__(INIT_WARPS * 32, GIBBS_INIT_MIN_BLOCKS) init_kernel(const ChainArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = a.s.n, k = a.k, row_words = a.s.row_words;
    uint32_t *lut = reinterpret_cast<uint32_t *>(smem_raw);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw + 64) + warp * 2;
    WarpTables WT;
    {
        unsigned char *b = smem_raw + 64 + INIT_WARPS * 16 + warp * WARP_TABLE_BYTES;
        WT.wcol = reinterpret_cast<double *>(b);
        WT.ptab = reinterpret_cast<int32_t *>(b + 1024);
        WT.lgcol = reinterpret_cast<int32_t *>(b + 2048);
        WT.counts = reinterpret_cast<int32_t *>(b + 2560);
    }
    require_aligned_tables(WT);
    uint32_t *rows = reinterpret_cast<uint32_t *>(smem_raw + 64 + INIT_WARPS * 16 + INIT_WARPS * WARP_TABLE_BYTES) +
                     warp * 2 * row_words;
    if (tid < 16) lut[tid] = hist_lut_entry(tid);
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_barrier_init();
    }
    __syncthreads();

    const long long total = (long long)a.n_chains * N;
    const long long stride = (long long)gridDim.x * INIT_WARPS;
    long long item = (long long)blockIdx.x * INIT_WARPS + warp;
    const uint32_t bytes = (uint32_t)row_words * 4u;
    auto issue = [&](long long it, uint32_t v) {
        if (lane == 0) {
            const int slot = (int)(v & 1u);
            mbar_expect_tx(bar + slot, bytes);
            bulk_g2s(rows + slot * row_words, a.s.packed + (size_t)(it % N) * row_words, bytes, bar + slot);
        }
    };
    unsigned long long st_updates = 0, st_windows = 0, st_slow = 0;
    uint32_t v = 0;
    if (item < total) issue(item, 0);
    while (item < total) {
        const long long next = item + stride;
        if (next < total) issue(next, v + 1); // the other slot was released by the __syncwarp below
        mbar_wait(bar + (v & 1u), (v >> 1) & 1u);
        const uint32_t *row = rows + (v & 1u) * row_words;
        const int chain = (int)(item / N), n = (int)(item % N);
        const int Wn = __ldg(a.s.len + n) - k + 1;
        random_loo_counts_impl<KP, (KP <= 6 ? GIBBS_P0_NB_INIT_SMALL : GIBBS_P0_NB_INIT_LARGE), false>(a, (uint64_t)a.chain_id_base + (uint64_t)chain, chain, n, WT.counts, lane, WT.lgcol);
        double p;
        int w;
        bool slow;
        if constexpr (DRIFT) {
            int f0[4], cn[4];
            const bool given = a.ppm_given != nullptr;
            const bool fast = a.drift_fast_ok && !given;
            drift_tables<KP>(WT, WT.counts, false, 0, k, a, given, fast, n, lane, f0, cn);
            slow = drift_pick<KP>(WT, row, Wn, k, a, fast, f0, cn, lane, p, w, -1, n);
        } else {
            build_tables<KP>(WT, WT.counts, false, 0, k, a.wtab, lane);
            slow = pick_argmax<KP>(WT, row, Wn, k, a.fast_ok, lane, p, w); // (sets with masked symbols never get here)
        }
        if (lane == 0) {
            a.sites[(size_t)chain * N + n] = w;
            a.hv[(size_t)chain * N + n] = p;
        }
        st_updates += 1;
        st_windows += (unsigned long long)Wn;
        st_slow += slow ? 1 : 0;
        __syncwarp();
        item = next;
        ++v;
    }
    if (lane == 0) {
        atomicAdd(a.stats + ST_SITE_UPDATES, st_updates);
        atomicAdd(a.stats + ST_WINDOW_SCORES, st_windows);
        atomicAdd(a.stats + ST_EXACT_RESCANS, st_slow);
    }
    if (blockIdx.x == 0 && tid == 0) atomicAdd(a.stats + ST_SWEEPS, (unsigned long long)a.n_chains);
}

// ------------------------------------------------------------------------------------------------
// random starts with the whole packed set resident in shared memory
// ------------------------------------------------------------------------------------------------
// The N(N-1) draws of a restart gather a k-mer at a random position of every other sequence. From global memory that
// is 2-3 L1 sector requests per draw, each a wavefront of its own (random rows); when the packed set fits beside the
// per-warp tables (C2: 144 KB of 227 KB) one CTA per SM keeps a copy in shared memory and the gathers become LDS with
// a few-way bank conflict. One warp per (chain, held-out sequence) item, grid-stride; the held-out row is scanned from
// the same copy, so this kernel issues no TMA at all.
#ifndef GIBBS_ISM_WARPS
#define GIBBS_ISM_WARPS 24 // 80 registers per thread: no spills at k <= 12 (32 warps / 64 registers spill)
#endif
#ifndef GIBBS_P0_NB_ISM
#define GIBBS_P0_NB_ISM 1  // LDS latency is short: one Philox block (4 gathers) in flight per lane is enough
#endif
constexpr int ISM_WARPS = GIBBS_ISM_WARPS;

// per-warp tables sized for the k at hand: wcol 64 KP + ptab 64 KP + lgcol 32 KP + counts 32 KP bytes
__host__ __device__ constexpr int ism_table_bytes(int kp) { return 192 * kp; }
__host__ __device__ inline size_t init_smem_rows_bytes(int n, int row_words) { return ((size_t)n * row_words * 4 + 63) / 64 * 64; }
__host__ __device__ inline size_t init_smem_total_bytes(int n, int row_words, int kp) {
    return init_smem_rows_bytes(n, row_words) + (size_t)ISM_WARPS * ism_table_bytes(kp);
}

template <int KP>
static __global__ void __launch_bounds__(ISM_WARPS * 32, 1) init_smem_kernel(const ChainArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = a.s.n, k = a.k, row_words = a.s.row_words;
    uint32_t *rows = reinterpret_cast<uint32_t *>(smem_raw);
    WarpTables WT;
    {
        unsigned char *b = smem_raw + init_smem_rows_bytes(N, row_words) + warp * ism_table_bytes(KP);
        WT.wcol = reinterpret_cast<double *>(b);
        WT.ptab = reinterpret_cast<int32_t *>(b + 64 * KP);
        WT.lgcol = reinterpret_cast<int32_t *>(b + 128 * KP);
        WT.counts = reinterpret_cast<int32_t *>(b + 160 * KP);
    }
    require_aligned_tables(WT);
    {   // rows are multiples of 16 B
        const uint4 *src = reinterpret_cast<const uint4 *>(a.s.packed);
        uint4 *dst = reinterpret_cast<uint4 *>(rows);
        const int n16 = N * (row_words >> 2);
        for (int i = tid; i < n16; i += ISM_WARPS * 32) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    const long long total = (long long)a.n_chains * N;
    const long long stride = (long long)gridDim.x * ISM_WARPS;
    unsigned long long st_updates = 0, st_windows = 0, st_slow = 0;
    for (long long item = (long long)blockIdx.x * ISM_WARPS + warp; item < total; item += stride) {
        const int chain = (int)(item / N), n = (int)(item % N);
        const int Wn = __ldg(a.s.len + n) - k + 1;
        random_loo_counts_impl<KP, GIBBS_P0_NB_ISM, false, true>(a, (uint64_t)a.chain_id_base + (uint64_t)chain, chain, n, WT.counts,
                                                                 lane, WT.lgcol, rows);
        build_tables<KP>(WT, WT.counts, false, 0, k, a.wtab, lane);
        double p;
        int w;
        const bool slow = pick_argmax<KP>(WT, rows + (size_t)n * row_words, Wn, k, a.fast_ok, lane, p, w);
        if (lane == 0) {
            a.sites[(size_t)chain * N + n] = w;
            a.hv[(size_t)chain * N + n] = p;
        }
        st_updates += 1;
        st_windows += (unsigned long long)Wn;
        st_slow += slow ? 1 : 0;
        __syncwarp();
    }
    if (lane == 0) {
        atomicAdd(a.stats + ST_SITE_UPDATES, st_updates);
        atomicAdd(a.stats + ST_WINDOW_SCORES, st_windows);
        atomicAdd(a.stats + ST_EXACT_RESCANS, st_slow);
    }
    if (blockIdx.x == 0 && tid == 0) atomicAdd(a.stats + ST_SWEEPS, (unsigned long long)a.n_chains);
}

// ------------------------------------------------------------------------------------------------
// random starts of LARGE sets: the packed set streamed through shared memory in tiles
// ------------------------------------------------------------------------------------------------
// C4 (100 000 x 200 bp) draws N (N - 1) = 1e10 sites per restart. From global memory every draw is a gather at a random
// address: one L1 sector per lane, and the L1 tag stage takes about one sector per cycle per SM -- 148 x 1.965 GHz =
// 2.9e11 draws/s whatever else the kernel does (init_kernel with the 64-bit gather copy measures 2.84e11, l1tex
// throughput 75 %, 0.87 sectors per cycle per SM: profiles/r02_ncu_init_wide.txt). Shared memory takes a random gather
// per lane at a few-way bank conflict instead, so the set is cut into tiles of `tile_rows` sequences that pass through
// two shared-memory buffers (cp.async.bulk, one mbarrier each): one CTA per SM, one (chain, held-out sequence) item per
// warp, all warps of the CTA on the same tile at the same time. A tile holds the sequences i0 <= i < i1, i.e. the draws
// of ranks [i0 - (i0 > n), i1 - (i1 > n)) of item (chain, n) (rank = position of i among the sequences other than n,
// fs:419-421) -- a contiguous range of the item's Philox stream, so the bit-sliced counters (KmerCounter) simply stay
// in registers from tile to tile. Philox blocks cut by a tile edge are computed on both sides (2 of ~275 per tile).
// After the last tile the warp scans its own sequence, staged from global memory, exactly like the other init kernels.
#ifndef GIBBS_TILED_WARPS
#define GIBBS_TILED_WARPS 16 // 128 registers per thread: the counters of k > 16 (36 registers) and a Philox block without spills
#endif
constexpr int TILED_WARPS = GIBBS_TILED_WARPS;
#ifndef GIBBS_TILED_NB
#define GIBBS_TILED_NB 1 // Philox blocks per lane and loop iteration
#endif

template <int KP, bool UNI>
__device__ __forceinline__ void tile_draws(const ChainArgs &a, const PhiloxKeys &pk, uint64_t chain_uid, uint64_t base, int n, int ra,
                                           int rb, int i0, const uint32_t *tile, uint32_t range_u, KmerCounter<KP> &h, int &since,
                                           bool &first, int32_t *counts, int lane) {
    using Word = typename KmerCounter<KP>::Word;
    const int k = a.k, row_words = a.s.row_words;
    const uint64_t blkA = (base + (uint64_t)ra) >> 2, blkB = (base + (uint64_t)rb + 3) >> 2;
    const int n_blk = (int)(blkB - blkA);
    constexpr int NB = GIBBS_TILED_NB;
    const int iters = (n_blk + 32 * NB - 1) / (32 * NB);
    const int r_first = (int)((int64_t)(blkA << 2) - (int64_t)base); // rank of draw 0 of block blkA (may lie before ra)
    const unsigned span = (unsigned)(rb - ra);
    // Plain blocks: all four draws belong to this tile and lie on one side of the held-out sequence, so they visit four
    // consecutive rows of the tile -- no validity test, no skip of n per draw. They are the blocks [lo_blk, hi_blk) except
    // the one that straddles n (hole_blk); an iteration whose 32 NB blocks are all plain (or past the end, when the last
    // block is whole) takes the short path. Warp-uniform arithmetic, nothing per lane.
    const int lo_blk = r_first == ra ? 0 : 1;
    const int hi_blk = (rb - r_first) >> 2; // blocks that end at or before rb
    const int hole_off = n - r_first;       // rank n relative to block 0: a block straddles n iff n is not at its start
    const int hole_blk = (hole_off > 0 && (hole_off & 3) != 0) ? (hole_off >> 2) : -1;
    for (int it = 0; it < iters; ++it) {
        // NB Philox blocks per lane and iteration: independent dependency chains for the few warps of this kernel
        int r0[NB];
        bool act[NB];
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            const int bi = (it * NB + q) * 32 + lane;
            r0[q] = r_first + 4 * bi;
            act[q] = bi < n_blk;
        }
        const int b_first = it * NB * 32, b_last = b_first + NB * 32; // this iteration's blocks [b_first, b_last)
        const bool plain = b_first >= lo_blk && (b_last <= hi_blk || hi_blk == n_blk) && !(hole_blk >= b_first && hole_blk < b_last);
        Word kmer[NB][4];
        if (plain) {
#pragma unroll
            for (int q = 0; q < NB; ++q) {
#pragma unroll
                for (int x = 0; x < 4; ++x) kmer[q][x] = 0;
                if (act[q]) {
                    const uint64_t blk = blkA + (uint64_t)((it * NB + q) * 32 + lane);
                    const uint4 r4 = philox4x32_10_keyed(make_uint4((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)chain_uid, (uint32_t)(chain_uid >> 32)), pk);
                    const uint32_t wd[4] = {r4.x, r4.y, r4.z, r4.w};
                    const int ib = r0[q] + (r0[q] >= n ? 1 : 0) - i0;
#pragma unroll
                    for (int x = 0; x < 4; ++x) {
                        const uint32_t range = UNI ? range_u : (uint32_t)(__ldg(a.s.len + i0 + ib + x) - k + 1);
                        const int pos = (int)__umulhi(wd[x], range); // floor(word * 2^-32 * range), exact
                        kmer[q][x] = gather_kmer<KP, true>(tile, row_words, ib + x, pos);
                    }
                }
            }
        } else {
#pragma unroll
            for (int q = 0; q < NB; ++q) {
                const uint64_t blk = blkA + (uint64_t)((it * NB + q) * 32 + lane);
                const uint4 r4 = philox4x32_10_keyed(make_uint4((uint32_t)blk, (uint32_t)(blk >> 32), (uint32_t)chain_uid, (uint32_t)(chain_uid >> 32)), pk);
                const uint32_t wd[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const bool ok = (unsigned)(r0[q] + x - ra) < span; // the draw belongs to this tile (and to the item at all)
                    const int r = ok ? r0[q] + x : ra;
                    const int i = r + (r >= n ? 1 : 0);
                    const uint32_t range = UNI ? range_u : (uint32_t)(__ldg(a.s.len + i) - k + 1);
                    const int pos = (int)__umulhi(wd[x], range);
                    const Word km = gather_kmer<KP, true>(tile, row_words, i - i0, pos);
                    kmer[q][x] = ok ? km : (Word)0;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < NB; ++q) {
            h.add4(kmer[q]);
            if (++since == 63) { // 252 k-mers per lane: the byte fields are full
                h.flush(counts, k, 0, first, lane);
                first = false;
                since = 0;
            }
        }
    }
}

__host__ __device__ inline size_t init_tiled_tile_bytes(int tile_rows, int row_words) { return ((size_t)tile_rows * row_words * 4 + 127) / 128 * 128; }
__host__ __device__ inline size_t init_tiled_total_bytes(int tile_rows, int row_words, int kp) {
    return 128 + 2 * init_tiled_tile_bytes(tile_rows, row_words) + (size_t)TILED_WARPS * (ism_table_bytes(kp) + (size_t)row_words * 4);
}

template <int KP>
static __global__ void __launch_bounds__(TILED_WARPS * 32, 1) init_tiled_kernel(const ChainArgs a, int tile_rows, const PhiloxKeys pk) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = a.s.n, k = a.k, row_words = a.s.row_words;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    const size_t tile_bytes = init_tiled_tile_bytes(tile_rows, row_words);
    uint32_t *tiles = reinterpret_cast<uint32_t *>(smem_raw + 128);
    unsigned char *wbase = smem_raw + 128 + 2 * tile_bytes;
    WarpTables WT;
    {
        unsigned char *b = wbase + warp * ism_table_bytes(KP);
        WT.wcol = reinterpret_cast<double *>(b);
        WT.ptab = reinterpret_cast<int32_t *>(b + 64 * KP);
        WT.lgcol = reinterpret_cast<int32_t *>(b + 128 * KP);
        WT.counts = reinterpret_cast<int32_t *>(b + 160 * KP);
    }
    require_aligned_tables(WT);
    uint32_t *own_row = reinterpret_cast<uint32_t *>(wbase + (size_t)TILED_WARPS * ism_table_bytes(KP)) + warp * row_words;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        fence_barrier_init();
    }
    __syncthreads();

    const long long total = (long long)a.n_chains * N;
    const long long per_batch = (long long)gridDim.x * TILED_WARPS;
    const long long first_item = (long long)blockIdx.x * TILED_WARPS;
    const int n_tiles = (N + tile_rows - 1) / tile_rows;
    const long long n_batches = first_item < total ? (total - first_item + per_batch - 1) / per_batch : 0;
    const long long total_q = n_batches * n_tiles;
    auto issue = [&](long long q) { // thread 0: tile q % n_tiles into buffer q & 1
        const int t = (int)(q % n_tiles);
        const int r0 = t * tile_rows, r1 = min(N, r0 + tile_rows);
        const uint32_t bytes = (uint32_t)(r1 - r0) * (uint32_t)row_words * 4u;
        uint64_t *b = bar + (q & 1);
        unsigned char *dst = reinterpret_cast<unsigned char *>(tiles) + (q & 1) * tile_bytes;
        const unsigned char *src = reinterpret_cast<const unsigned char *>(a.s.packed + (size_t)r0 * row_words);
        mbar_expect_tx(b, bytes);
        for (uint32_t o = 0; o < bytes; o += 32768u) bulk_g2s(dst + o, src + o, min(32768u, bytes - o), b);
    };
    const uint32_t range_u = (uint32_t)(a.s.uniform_len - k + 1);
    unsigned long long st_updates = 0, st_windows = 0, st_slow = 0;
    KmerCounter<KP> h;
    h.clear();
    int since = 0, chain = 0, n = 0, t = 0;
    bool first = true, valid = false;
    uint64_t base = 0, chain_uid = 0;
    long long batch = 0;
    if (tid == 0 && total_q > 0) issue(0);
    for (long long q = 0; q < total_q; ++q) {
        if (tid == 0 && q + 1 < total_q) issue(q + 1); // its buffer was released by the barrier that ended tile q - 1
        if (t == 0) { // a new batch: this warp's item
            const long long item = first_item + batch * per_batch + warp;
            valid = item < total;
            if (valid) {
                chain = (int)(item / N);
                n = (int)(item % N);
                chain_uid = (uint64_t)a.chain_id_base + (uint64_t)chain;
                base = (uint64_t)n * (uint64_t)(N - 1);
                for (int i = lane; i < row_words; i += 32) own_row[i] = __ldg(a.s.packed + (size_t)n * row_words + i);
            }
            h.clear();
            since = 0;
            first = true;
        }
        mbar_wait(bar + (q & 1), (uint32_t)((q >> 1) & 1));
        if (valid) {
            const int i0 = t * tile_rows, i1 = min(N, i0 + tile_rows);
            const int ra = i0 - (i0 > n ? 1 : 0), rb = i1 - (i1 > n ? 1 : 0);
            const uint32_t *tile = reinterpret_cast<const uint32_t *>(reinterpret_cast<const unsigned char *>(tiles) + (q & 1) * tile_bytes);
            if (rb > ra) {
                if (a.s.uniform_len > 0) tile_draws<KP, true>(a, pk, chain_uid, base, n, ra, rb, i0, tile, range_u, h, since, first, WT.counts, lane);
                else tile_draws<KP, false>(a, pk, chain_uid, base, n, ra, rb, i0, tile, range_u, h, since, first, WT.counts, lane);
            }
        }
        __syncthreads(); // every warp is done with this buffer
        if (++t == n_tiles) {
            t = 0;
            ++batch;
            if (valid) {
                h.flush(WT.counts, k, N - 1, first, lane);
                KmerCounter<KP>::finish(WT.counts, k, lane);
                const int Wn = __ldg(a.s.len + n) - k + 1;
                build_tables<KP>(WT, WT.counts, false, 0, k, a.wtab, lane);
                double p;
                int w;
                const bool slow = pick_argmax<KP>(WT, own_row, Wn, k, a.fast_ok, lane, p, w);
                if (lane == 0) {
                    a.sites[(size_t)chain * N + n] = w;
                    a.hv[(size_t)chain * N + n] = p;
                }
                st_updates += 1;
                st_windows += (unsigned long long)Wn;
                st_slow += slow ? 1 : 0;
                __syncwarp();
            }
        }
    }
    if (lane == 0) {
        atomicAdd(a.stats + ST_SITE_UPDATES, st_updates);
        atomicAdd(a.stats + ST_WINDOW_SCORES, st_windows);
        atomicAdd(a.stats + ST_EXACT_RESCANS, st_slow);
    }
    if (blockIdx.x == 0 && tid == 0) atomicAdd(a.stats + ST_SWEEPS, (unsigned long long)a.n_chains);
}

// ------------------------------------------------------------------------------------------------
// the chain kernel: one team (CTA of T warps) = one restart of SiteSampler.doSiteSamplingWithBPV
// (fs:691-695)
// ------------------------------------------------------------------------------------------------
// A ROUND = T consecutive held-out sequences n0 .. n0+T-1, one per warp, scored concurrently.
//   random starts (fs:412) and shift sweeps (fs:350 / fs:318): every site update of a sweep reads
//     the same snapshot, so all T results of a round are committed.
//   greedy sweeps (fs:381) are in-place: sequence n must see the sites accepted for 0..n-1. The round
//     is speculative: results are committed in order up to and including the first warp whose accepted
//     update MOVES a site (that changes the counts); later warps of the round are discarded and redone
//     in the next round, which starts right after the mover. The committed sequence of site updates is
//     therefore exactly the reference's sequential sweep.
// MASKED = the set holds symbols outside A,C,G,T (a.s.mask != null): a separate instantiation (4 warps only), because
// the 4-warp kernel sits at its register limit and even never-taken branches cost the ACGT path 2-3 %.
// DRIFT = the data-derived background of doSiteSampling (fs:697): same sweeps, rounds and hand-over; the site update
// builds the PPM instead of the odds table and scans with the per-window background (gibbs_drift_dev.cuh). Same launch
// bounds (measured on C2: 7 CTAs of 4 warps at 72 registers 166 ms, 6 at 80 178 ms, 4 at 118 registers 185-193 ms).
// INIT_ONLY = the instantiation that runs the random starts (fs:412) on the chain's own team and nothing else; the
// sweep instantiations (INIT_ONLY = false) contain no random-start code at all, so the register-limited 4-warp kernel
// pays nothing for a phase that a grid-wide kernel normally runs (gibbs_api.cu, launch_random_starts).
template <int KP, int T, bool MASKED = false, bool DRIFT = false, bool INIT_ONLY = false>
static __global__ void __launch_bounds__(32 * T, (INIT_ONLY ? (T == 1 ? 8 : 4) : T == 1 ? 16 : T == 4 ? GIBBS_T4_MIN_BLOCKS : T == 8 ? GIBBS_T8_MIN_BLOCKS : GIBBS_T16_MIN_BLOCKS)) chain_kernel(const ChainArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int THREADS = 32 * T;
    constexpr int R = (2 * T < 4) ? 4 : 2 * T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int chain = blockIdx.x;
    if (a.from_list) { // continuing paused chains: one CTA per list entry
        if ((int)blockIdx.x >= *a.pending_in_n) return;
        chain = a.pending_in[blockIdx.x];
    }
#include "gibbs_chain_body.inc" // (shared with chain_batch_kernel, gibbs_batch.cuh)
}

// ------------------------------------------------------------------------------------------------
// primitive kernels (one warp): same device routines as the chain kernel
// ------------------------------------------------------------------------------------------------
struct PrimArgs {
    DeviceSeqs s;
    const WEnt *wtab;
    const int32_t *sites; // [n] device
    int32_t heldout;
    int32_t k;
    int32_t fast_ok;
    int32_t *counts_out;  // [k*4]
    double *raw_out;      // [W] or null
    double *log2_out;     // [W] or null
    double *score_out;    // [2]: log2 max, raw max
    int32_t *site_out;    // [2]: argmax, used_exact_rescan
};

template <int KP>
static __global__ void __launch_bounds__(32) loo_counts_kernel(const PrimArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    const TeamSmem S = carve_smem(smem_raw, 1);
    if (lane < 16) S.lut[lane] = hist_lut_entry(lane);
    __syncwarp();
    site_counts<KP, 1>(a.s, a.sites, a.heldout, a.k, SHIFT_NONE, S.total, S.lut, S.fix, lane);
    for (int e = lane; e < a.k * 4; e += 32) a.counts_out[e] = S.total[e];
}

// mode 0: every window in float64 (raw product and log2); mode 1: argmax pick
template <int KP>
static __global__ void __launch_bounds__(32) scan_kernel(const PrimArgs a, int mode) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    const TeamSmem S = carve_smem(smem_raw, 1);
    const WarpTables WT = warp_tables(S, 0);
    require_aligned_tables(WT);
    RowRing<4> ring;
    ring.init(S, a.s, a.heldout, lane);
    if (lane < 16) S.lut[lane] = hist_lut_entry(lane);
    __syncwarp();
    if (lane == 0) ring.fill(1);
    site_counts<KP, 1>(a.s, a.sites, a.heldout, a.k, SHIFT_NONE, S.total, S.lut, S.fix, lane);
    const uint32_t *row = ring.wait(0);
    build_tables<KP>(WT, S.total, false, 0, a.k, a.wtab, lane);
    const int W = __ldg(a.s.len + a.heldout) - a.k + 1;
    const int masked_n = row_masked(a.s, a.heldout) ? a.heldout : -1;
    if (mode == 0) {
        for (int w = lane; w < W; w += 32) {
            double p = exact_window<KP>(row, w, a.k, WT.wcol);
            if (masked_n >= 0 && mask_kmer(a.s.mask, a.s.row_words, masked_n, w, a.k) != 0) p = 0.0; // PWM row of the symbol is 0
            if (a.raw_out) a.raw_out[w] = p;
            if (a.log2_out) a.log2_out[w] = log2_ref(p);
        }
    } else {
        double p;
        int w;
        const bool slow = pick_argmax<KP>(WT, row, W, a.k, a.fast_ok, lane, p, w, &a.s, masked_n);
        if (lane == 0) {
            a.score_out[0] = log2_ref(p);
            a.score_out[1] = p;
            a.site_out[0] = w;
            a.site_out[1] = slow ? 1 : 0;
        }
    }
}

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

// first chain with the largest sum (strict >), the restart selection of fs:450 / fs:156-170: what the sequential
//   best = 0; for c = 1 ..: if sums[c] > sums[best] then best = c
// returns (a NaN sum never wins a comparison; with sums[0] = NaN nothing beats it). One CTA.
static __global__ void __launch_bounds__(256) best_chain_kernel(const double *sums, int n_chains, int *best_out) {
    __shared__ double s_v[256];
    __shared__ int s_i[256];
    double bv = -INFINITY;
    int bi = INT32_MAX;
    for (int c = threadIdx.x; c < n_chains; c += 256) {
        const double v = sums[c];
        if (v > bv || (v == bv && c < bi)) { // ascending c per thread: ties keep the lowest index
            bv = v;
            bi = c;
        }
    }
    s_v[threadIdx.x] = bv;
    s_i[threadIdx.x] = bi;
    __syncthreads();
    for (int o = 128; o; o >>= 1) {
        if ((int)threadIdx.x < o) {
            const double ov = s_v[threadIdx.x + o];
            const int oi = s_i[threadIdx.x + o];
            if (ov > s_v[threadIdx.x] || (ov == s_v[threadIdx.x] && oi < s_i[threadIdx.x])) {
                s_v[threadIdx.x] = ov;
                s_i[threadIdx.x] = oi;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double s0 = sums[0];
        // every sum NaN or -inf: nothing is > sums[0]
        *best_out = (s0 != s0 || s_i[0] == INT32_MAX || !(s_v[0] > s0)) ? 0 : s_i[0];
    }
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
#include "gibbs_restart_select_body.inc" // (shared with restart_select_batch_kernel, gibbs_batch.cuh)
}

// element `which` of every Positions pair: the site arrays the one-site kernels take
static __global__ void pair_element_kernel(const int32_t *pos2, int n, int which, int32_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = pos2[2 * i + which];
}

// ------------------------------------------------------------------------------------------------
// shared-memory streaming microbenchmark: the measured denominator of the smem roofline
// ------------------------------------------------------------------------------------------------
// 1024 threads x LDS.128, conflict-free, 8 loads per round: bytes = grid * 1024 * 16 * 8 * iters
static __global__ void __launch_bounds__(1024) smem_stream_kernel(int iters, unsigned int *sink) {
    __shared__ uint4 buf[2048];
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) buf[i] = make_uint4(i, i * 3, i * 5, i * 7);
    __syncthreads();
    uint4 acc = make_uint4(0, 0, 0, 0);
    int idx = threadIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint4 v = buf[idx];
            acc.x ^= v.x; acc.y += v.y; acc.z ^= v.z; acc.w += v.w;
            idx = (idx + 1024 + 32) & 2047;
        }
    }
    if ((acc.x ^ acc.y ^ acc.z ^ acc.w) == 0x9e3779b9u) *sink = 1;
}

} // namespace gibbs
