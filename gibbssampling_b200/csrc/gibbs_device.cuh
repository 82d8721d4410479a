// gibbssampling_b200/csrc/gibbs_device.cuh -- device-side building blocks (sm_100a only).
//
// A team of T warps (one CTA) owns one chain (= one restart of the reference, fs:691-695). The unit
// of work is one SITE UPDATE (leave-one-out PWM -> score every window of the held-out sequence ->
// pick), and one WARP does a whole site update: its k x 4 PWM column table (float64), its
// fixed-point log2-odds pair table and the 2-bit packed row it scans live in shared memory. The T
// warps of a team work on T consecutive held-out sequences at once (see gibbs_kernels.cuh).
//
// Exactness strategy (DESIGN.md "Kernels"): every window is first scored with an int32
// fixed-point sum of log2-odds looked up two bases at a time (one LDS + half an IADD3 per
// column pair). That ranks windows up to a rigorous rounding margin; the few windows inside the
// margin of the maximum are re-scored with the reference's own arithmetic -- a left-to-right
// float64 product of odds ratios (fs:290-293) -- so the argmax and its score are bit-identical
// to the reference's float64 scan (fs:301-314).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

namespace gibbs {

constexpr unsigned FULL = 0xffffffffu;
constexpr int LG_FRAC_BITS = 11;          // log2-odds fixed point: 2^-11 units ...
constexpr int KEY_IDX_BITS = 8;           // ... shifted left by 8 to leave room for a window index
constexpr int MAX_COLS = 32;              // GIBBS_MAX_K
constexpr double LN2 = 0.6931471805599453; // log 2.0 as float64 (FSharpAux log2 = ln x / ln 2)

enum ShiftMode { SHIFT_NONE = 0, SHIFT_LEFT = 1, SHIFT_RIGHT = 2 };
enum StatSlot { ST_SITE_UPDATES = 0, ST_WINDOW_SCORES = 1, ST_SWEEPS = 2, ST_EXACT_RESCANS = 3, ST_CAPPED = 4,
                ST_SPECULATED = 5, ST_NSLOTS = 8 };

// one entry per (count, base): the odds ratio W = ((c + pc) / den) / q[b] of fs:260 + fs:286 as
// float64, and round(log2 W * 2^11) << 8 for the ranking pass
struct __align__(16) WEnt {
    double w;
    int32_t lg;
    int32_t pad;
};

struct DeviceSeqs {
    const uint32_t *packed; // [n][row_words], base b of a row in bits [2(b%16), +2) of word b/16
    const int32_t *len;     // [n]
    int32_t n;
    int32_t row_words;      // multiple of 4 (16 B) and >= ceil(max_len/16) + 4 zero words
    int32_t uniform_len;    // > 0: every sequence has this length (saves a dependent load per random draw)
    // Symbols outside A,C,G,T (IUPAC codes, Gap, Ter: any index the reference's 49-slot tables accept but
    // whose PWM row is 0 because it is not in `alphabet`, fs:283-287). Null when the set has none, so the
    // pure-ACGT path pays one uniform branch. mask has the geometry of `packed` with 0b01 at Gap '-' and 0b11 at
    // the other such symbols (their 2-bit code is 0): bit 0 marks every symbol outside A,C,G,T, bit 1 tells Gap
    // from the rest (read only where Gap is a member of the alphabet); rowflag[i] != 0 iff sequence i holds one.
    const uint32_t *mask;
    const int32_t *rowflag;
    // Gather copy for the random starts of sets that do not fit shared memory: wide[i][m] = the 32 bases from base 8 m of
    // sequence i as one 64-bit word (windows overlap: 4x the packed size). A k-mer of k <= 25 at ANY position is one aligned
    // 8-byte load -- one L1 sector request per draw instead of the two or three 4-byte requests of the packed rows.
    const uint64_t *wide;
    int32_t wide_words;     // words per sequence: max_len / 8 + 1
};

struct ChainArgs {
    DeviceSeqs s;
    const WEnt *wtab;       // [n][4]
    int32_t k;
    int32_t max_sweeps;
    int32_t fast_ok;
    int32_t sampler;
    int32_t phase_mask;     // GIBBS_PHASE_* bits to run, in pipeline order
    int32_t rng_mode;       // 0 Philox, 1 injected
    uint64_t seed;
    int64_t chain_id_base;
    const double *uniforms;
    int64_t uniforms_per_chain;
    int32_t n_chains;
    int32_t *sites;         // [chains][n]
    double *hv;             // [chains][n] raw float64 score (odds product or background product)
    double *scores;         // [chains][n] log2 / PWMS
    double *sums;           // [chains]
    unsigned long long *stats;
    double cutoff;
    double bg[4];
    // getMotifsWithBestPWMSOfPPM (fs:644-661): the random starts are scored against this caller-supplied PPM
    // ([k][4], rows A,C,G,T of the reference's 49 x k matrix) instead of the PPM of the random sites; the random sites
    // then only shape the background. Null = the usual random starts. Data-derived background only.
    const double *ppm_given;
    // data-derived background (chain_kernel<.., DRIFT = true>, fs:462-640): normalizePPM value of a count
    // (c + pc) / ((N-1) + |A| pc) (fs:260), base counts per sequence and of the whole set, |A| pc (fs:117)
    const double *pvals;      // [n]
    const int32_t *basecnt;   // [n][4]
    const int32_t *maskcnt;   // [n] symbols outside A,C,G,T per sequence (null when the set has none)
    int32_t gcnt[4];
    double alpha_pc, pc;
    int32_t drift_fast_ok;    // the float32 ranking pass may be used
    // Gaps '-' of the set when Gap is a member of the alphabet (SiteSampler, data-derived background, alphabet_size >= 5),
    // else 0: Gap is then a dead symbol like N. Read by the MASKED instantiations only; it fills the padding before `ss`,
    // so the layout of ChainArgs (and the code of every other instantiation) is unchanged.
    int32_t gap_total;
    const int32_t *ss;        // [n][ss_stride][4] prefix tables of every sequence (prefix_kernel), or null
    int32_t ss_stride;        // entries (int4) per sequence: max_len + 2
    // pause / resume at sweep boundaries: once few chains are still running they are continued by a
    // following launches with wider teams: 4 -> 8 -> 16 warps per chain (see launch_chain_kp)
    // greedy sweeps: narrowest speculative round. 1 while many chains share an SM (discarded work costs the others issue
    // slots); the team size once a chain has its SM(s) to itself -- idle warps are free, only latency counts there
    int32_t min_width;
    int32_t *active;          // chains not finished yet
    int32_t pause_below;      // pause when *active <= pause_below (0 = never)
    int32_t pause_min_sweeps; // ... and the chain has run at least this many sweeps in this launch (chain_kernel only)
    int32_t from_list;        // 1 = this launch continues the chains listed in pending_in
    int32_t *resume;          // [chains] phase | sweeps_in_phase << 8 of a paused chain
    const int32_t *pending_in;
    const int32_t *pending_in_n;
    int32_t *pending_out;
    int32_t *pending_out_n;
};

// ------------------------------------------------------------------------------------------------
// shared memory: per-warp tables + per-team state
// ------------------------------------------------------------------------------------------------
struct WarpTables {       // private to the warp that runs a site update
    double *wcol;         // [32*4] float64 odds per column, entry j*4+b
    int32_t *ptab;        // [16*16] pair table: ptab[p*16 + nib] = lgcol[2p][nib&3] + lgcol[2p+1][nib>>2]
    int32_t *lgcol;       // [32*4] fixed-point log2 odds per column
    int32_t *counts;      // [32*4] leave-one-out counts of the random-init phase
};
constexpr int WARP_TABLE_BYTES = 1024 + 1024 + 512 + 512;

struct TeamSmem {
    uint64_t *bar;        // [ring] mbarriers of the staged rows
    int32_t *total;       // [32*4] counts over ALL current sites of the chain
    int32_t *flags;       // [2][T] per-warp outcome of a round (double-buffered) + [2T] pause decision, T <= 16
    uint32_t *lut;        // [16] histogram increments per nibble (hist_lut_entry)
    int32_t *fix;         // [32] per column: masked bases the histogram counted as code 0 (see hist_fix)
    double *blk_hv;       // [2][32] state of two 32-sequence blocks
    int32_t *blk_site;    // [2][32]
    int32_t *blk_len;     // [2][32]
    unsigned char *warp_tables; // T x WARP_TABLE_BYTES
    uint32_t *row0;       // ring of staged rows, slot s at row0 + s * row_words
};

constexpr int MAX_TEAM = 16;
constexpr int MAX_RING = 2 * MAX_TEAM;
// bar 256, total 512, flags 160, blk_hv 512, blk_site 256, blk_len 256, lut 64, fix 128, pad to 16 B
constexpr int TEAM_FIXED_BYTES = 2176;
static_assert(MAX_RING * 8 + 512 + 160 + 512 + 256 + 256 + 64 + 128 <= TEAM_FIXED_BYTES, "fixed part of the team's shared memory");

__host__ __device__ constexpr int ring_slots(int team_warps) { return 2 * team_warps < 4 ? 4 : 2 * team_warps; }
__host__ __device__ inline int team_smem_bytes(int row_words, int team_warps) {
    return TEAM_FIXED_BYTES + team_warps * WARP_TABLE_BYTES + ring_slots(team_warps) * row_words * 4;
}

__device__ __forceinline__ TeamSmem carve_smem(unsigned char *base, int team_warps) {
    TeamSmem s;
    s.bar = reinterpret_cast<uint64_t *>(base);
    s.total = reinterpret_cast<int32_t *>(base + 256);
    s.flags = reinterpret_cast<int32_t *>(base + 768);
    s.blk_hv = reinterpret_cast<double *>(base + 928);
    s.blk_site = reinterpret_cast<int32_t *>(base + 1440);
    s.blk_len = reinterpret_cast<int32_t *>(base + 1696);
    s.lut = reinterpret_cast<uint32_t *>(base + 1952);
    s.fix = reinterpret_cast<int32_t *>(base + 2016);
    s.warp_tables = base + TEAM_FIXED_BYTES;
    s.row0 = reinterpret_cast<uint32_t *>(base + TEAM_FIXED_BYTES + team_warps * WARP_TABLE_BYTES);
    return s;
}

// The MASKED instantiations (1 or 4 warps: a ring of at most 8 barriers) keep the gap row of `total` -- Gaps per column
// over the current sites, [32] -- in the upper half of the barrier array, which their rings leave unused.
__device__ __forceinline__ int32_t *gap_row(const TeamSmem &s) { return reinterpret_cast<int32_t *>(s.bar + MAX_RING / 2); }
static_assert(MAX_RING / 2 * 8 >= 32 * 4, "gap row");

__device__ __forceinline__ WarpTables warp_tables(const TeamSmem &s, int warp) {
    unsigned char *b = s.warp_tables + warp * WARP_TABLE_BYTES;
    WarpTables t;
    t.wcol = reinterpret_cast<double *>(b);
    t.ptab = reinterpret_cast<int32_t *>(b + 1024);
    t.lgcol = reinterpret_cast<int32_t *>(b + 2048);
    t.counts = reinterpret_cast<int32_t *>(b + 2560);
    return t;
}

template <int T>
__device__ __forceinline__ void team_sync() {
    if (T == 1) __syncwarp();
    else __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier + 1-D bulk async copy (TMA, SASS UBLKCP)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// the ranking pass ORs nibble offsets into the pair-table address: every per-warp table block must be 64-byte aligned
__device__ __forceinline__ void require_aligned_tables(const WarpTables &t) {
    if ((smem_u32(t.ptab) & 63u) != 0) __trap();
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// Ring of staged rows. Visits are numbered 0, 1, 2, ... over the whole chain (visit v scans sequence
// (first + v) mod N: every sweep walks n = 0..N-1), visit v lives in slot v % R and completes phase
// (v / R) & 1 of that slot's mbarrier, so any warp can find and wait for its row from v alone (R is a
// power of two, so 32-bit wrap-around of v is harmless). One elected thread keeps the rows of visits
// [head, head + R) in flight with cp.async.bulk (TMA).
template <int R>
struct RowRing {
    static_assert((R & (R - 1)) == 0, "ring size must be a power of two");
    uint64_t *bar;
    uint32_t *row0;
    const uint32_t *gpacked;
    int row_words, n_seqs;
    uint32_t issued;  // visits [0, issued) have been requested   (meaningful on thread 0 only)
    int next_seq;     // sequence of visit `issued`                (thread 0 only)

    __device__ __forceinline__ void init(const TeamSmem &s, const DeviceSeqs &d, int first, int tid) {
        bar = s.bar;
        row0 = s.row0;
        gpacked = d.packed;
        row_words = d.row_words;
        n_seqs = d.n;
        issued = 0;
        next_seq = first;
        if (tid == 0) {
#pragma unroll
            for (int i = 0; i < R; ++i) mbar_init(bar + i, 1);
            fence_barrier_init();
        }
    }
    // thread 0 only: request the rows of visits [issued, upto)
    __device__ __forceinline__ void fill(uint32_t upto) {
        const uint32_t bytes = (uint32_t)row_words * 4u;
        while (issued != upto) {
            const int slot = (int)(issued & (R - 1));
            mbar_expect_tx(bar + slot, bytes);
            bulk_g2s(row0 + slot * row_words, gpacked + (size_t)next_seq * row_words, bytes, bar + slot);
            next_seq = next_seq + 1 < n_seqs ? next_seq + 1 : 0;
            ++issued;
        }
    }
    // Stateless variant for a whole warp: lane l < cnt requests visit first_visit + l, which reads sequence
    // (first_seq + l) mod n_seqs. A round of T committed visits costs one issue sequence instead of T, and
    // the caller derives first_visit / first_seq from its loop counters (no ring state in registers).
    __device__ __forceinline__ void fill_span(uint32_t first_visit, int first_seq, int cnt, int lane) const {
        if (lane < cnt) {
            const uint32_t bytes = (uint32_t)row_words * 4u;
            const int slot = (int)((first_visit + (uint32_t)lane) & (R - 1));
            int seq = first_seq + lane;
            if (seq >= n_seqs) seq %= n_seqs;
            mbar_expect_tx(bar + slot, bytes);
            bulk_g2s(row0 + slot * row_words, gpacked + (size_t)seq * row_words, bytes, bar + slot);
        }
    }
    __device__ __forceinline__ const uint32_t *wait(uint32_t v) const {
        const int slot = (int)(v & (R - 1));
        mbar_wait(bar + slot, (v / R) & 1u);
        return row0 + slot * row_words;
    }
};

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al.), the counter-based uniform stream; same constants as the oracle
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// The same block cipher with the ten round keys precomputed on the host (they depend on the seed alone) and passed as a
// kernel parameter: the round keys become constant-bank operands of the LOP3s instead of twenty registers or two IADDs
// per round (init_tiled_kernel runs at its register limit and on the integer pipe).
struct PhiloxKeys {
    uint32_t x[10], y[10];
};
inline PhiloxKeys philox_round_keys(uint64_t seed) {
    PhiloxKeys pk;
    uint32_t kx = (uint32_t)seed, ky = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) {
        pk.x[r] = kx;
        pk.y[r] = ky;
        kx += 0x9E3779B9u;
        ky += 0xBB67AE85u;
    }
    return pk;
}
__device__ __forceinline__ uint4 philox4x32_10_keyed(uint4 c, const PhiloxKeys &pk) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ pk.x[r], lo1, hi0 ^ c.w ^ pk.y[r], lo0);
    }
    return c;
}

// ------------------------------------------------------------------------------------------------
// 2-bit k-mer extraction
// ------------------------------------------------------------------------------------------------
// 64 bits starting at base `pos` of a row (global memory, read-only path)
template <int KP>
__device__ __forceinline__ uint64_t kmer_global(const uint32_t *__restrict__ rowp, int pos) {
    const uint32_t *p = rowp + (pos >> 4);
    const int sh = (pos & 15) * 2;
    const uint32_t w0 = __ldg(p), w1 = __ldg(p + 1);
    uint32_t lo = __funnelshift_r(w0, w1, sh), hi = w1 >> sh;
    if (KP > 8) {
        const uint32_t w2 = __ldg(p + 2);
        hi = __funnelshift_r(w1, w2, sh);
    }
    return ((uint64_t)hi << 32) | lo;
}
template <int KP>
__device__ __forceinline__ uint64_t kmer_shared(const uint32_t *rowp, int pos) {
    const uint32_t *p = rowp + (pos >> 4);
    const int sh = (pos & 15) * 2;
    const uint32_t w0 = p[0], w1 = p[1];
    uint32_t lo = __funnelshift_r(w0, w1, sh), hi = w1 >> sh;
    if (KP > 8) {
        const uint32_t w2 = p[2];
        hi = __funnelshift_r(w1, w2, sh);
    }
    return ((uint64_t)hi << 32) | lo;
}

__device__ __forceinline__ int shifted_site(int pos, int len, int k, int mode) {
    if (mode == SHIFT_LEFT) return pos > 0 ? pos - 1 : pos;             // fs:358
    if (mode == SHIFT_RIGHT) return pos <= len - k - 1 ? pos + 1 : pos; // fs:327
    return pos;
}

// ------------------------------------------------------------------------------------------------
// symbols outside A,C,G,T (rare path, kept out of line so the ACGT path keeps its registers)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool row_masked(const DeviceSeqs &s, int i) { return s.mask != nullptr && __ldg(s.rowflag + i) != 0; }

// 2 bits per column of the k-mer at `pos` of sequence i: 0b11 where the base is not A,C,G,T
static __device__ __noinline__ uint64_t mask_kmer(const uint32_t *__restrict__ mask, int row_words, int i, int pos, int k) {
    const uint32_t *p = mask + (size_t)i * row_words + (pos >> 4);
    const int sh = (pos & 15) * 2;
    const uint32_t w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2);
    const uint64_t m = ((uint64_t)__funnelshift_r(w1, w2, sh) << 32) | __funnelshift_r(w0, w1, sh);
    return k >= 32 ? m : (m & ((1ull << (2 * k)) - 1ull));
}

// The histogram counted every masked base of this k-mer as code 0 (A): note the columns in fix[] so the
// caller can take them out again. The reference counts such a base in its own (dead) row, fs:211-215.
static __device__ __noinline__ void hist_fix(const uint32_t *__restrict__ mask, int row_words, int i, int pos, int k, int32_t *fix) {
    uint64_t m = mask_kmer(mask, row_words, i, pos, k);
    while (m) {
        const int j = (__ffsll((long long)m) - 1) >> 1;
        atomicAdd(&fix[j], 1);
        m &= ~(3ull << (2 * j));
    }
}

// hist_fix, and the Gaps among those columns counted into gap[] (the gap row of the counts)
static __device__ __noinline__ void hist_fix_gap(const uint32_t *__restrict__ mask, int row_words, int i, int pos, int k, int32_t *fix,
                                                 int32_t *gap) {
    uint64_t m = mask_kmer(mask, row_words, i, pos, k);
    while (m) {
        const int j = (__ffsll((long long)m) - 1) >> 1;
        atomicAdd(&fix[j], 1);
        if (((m >> (2 * j)) & 3u) == 1u) atomicAdd(&gap[j], 1);
        m &= ~(3ull << (2 * j));
    }
}

// ------------------------------------------------------------------------------------------------
// per-thread packed histogram of k-mers (replaces createPFMOf + fusePositionFrequencyMatrices,
// fs:211-226)
// ------------------------------------------------------------------------------------------------
// Two columns per lookup: lut[nib] (16 words of shared memory) holds a 1 in the 4-bit field of base
// nib&3 of the even column (fields 0-3) and of base nib>>2 of the odd column (fields 4-7). Nibble
// counters spill into byte counters every 15 adds, byte counters into dst[] every 255 adds.
__device__ __forceinline__ uint32_t hist_lut_entry(int nib) { return (1u << (4 * (nib & 3))) | (1u << (16 + 4 * (nib >> 2))); }

template <int KP>
struct Hist {
    uint32_t c4[KP];      // 8 nibble counters per column pair
    uint32_t lo[KP];      // byte counters of fields 0,2,4,6
    uint32_t hi[KP];      // byte counters of fields 1,3,5,7
    int n4;               // adds since the last nibble spill
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int p = 0; p < KP; ++p) c4[p] = lo[p] = hi[p] = 0;
        n4 = 0;
    }
    __device__ __forceinline__ void spill4() {
#pragma unroll
        for (int p = 0; p < KP; ++p) {
            lo[p] += c4[p] & 0x0F0F0F0Fu;
            hi[p] += (c4[p] >> 4) & 0x0F0F0F0Fu;
            c4[p] = 0;
        }
        n4 = 0;
    }
    // add up to 4 k-mers; caller guarantees n4 + 4 <= 15 after spill handling below
    __device__ __forceinline__ void add(uint64_t kmer, const uint32_t *lut) {
#pragma unroll
        for (int p = 0; p < KP; ++p) c4[p] += lut[(uint32_t)(kmer >> (4 * p)) & 15u];
        ++n4;
    }
    __device__ __forceinline__ void maybe_spill(int upcoming) {
        if (n4 + upcoming > 15) spill4(); // uniform enough: n4 differs between lanes only at range edges
    }
    // at most 255 adds per thread since the last flush; dst[] += warp sums. Bytes are widened to
    // 16-bit fields (32 lanes x 255 < 65536) so one REDUX.SUM reduces two counters at once.
    // ATOMIC: several warps add into the same dst.
    template <bool ATOMIC>
    __device__ __forceinline__ void flush_add(int32_t *dst, int k, int lane) {
        spill4();
#pragma unroll
        for (int p = 0; p < KP; ++p) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                // q = 0: lo bytes 0,2 (base 0 of both columns); 1: lo bytes 1,3 (base 2);
                // q = 2: hi bytes 0,2 (base 1); 3: hi bytes 1,3 (base 3)
                const uint32_t src = (q < 2) ? lo[p] : hi[p];
                const uint32_t s = __reduce_add_sync(FULL, (src >> (8 * (q & 1))) & 0x00FF00FFu);
                const int b = (q == 0) ? 0 : (q == 1) ? 2 : (q == 2) ? 1 : 3;
                if (lane == ((4 * p + q) & 31)) {
                    const int e0 = (2 * p) * 4 + b, e1 = (2 * p + 1) * 4 + b;
                    const int32_t v0 = (int32_t)(s & 0xFFFFu), v1 = (int32_t)(s >> 16);
                    if (!ATOMIC) {
                        dst[e0] += v0;
                        if (2 * p + 1 < k) dst[e1] += v1;
                    } else {
                        atomicAdd(&dst[e0], v0);
                        if (2 * p + 1 < k) atomicAdd(&dst[e1], v1);
                    }
                }
            }
            lo[p] = hi[p] = 0;
        }
    }
};

// ------------------------------------------------------------------------------------------------
// bit-sliced base counters for the random starts (fs:418-426): no table lookups
// ------------------------------------------------------------------------------------------------
// A k-mer is 2 bits per column. f_b = a 1 in the even bit of every column whose base is b (b = 1, 2, 3: three LOP3;
// base 0 is what is left: count_0 = k-mers added - count_1 - count_2 - count_3). Four k-mers are added at once (one
// Philox block): f(x0) + f(x1) + f(x2) fits the 2-bit column fields, and together with f(x3) the even / odd columns go
// into 4-bit fields (8 per word), which take 3 such quads before they are spread into 8-bit fields (255 k-mers per
// lane between warp reductions). ~11 integer instructions per k-mer against ~45 for the pair-LUT histogram (6 shared
// loads + extraction per k-mer), which is what the random starts of a C2 step spent half their instructions on.
template <int KP>
struct KmerCounter {
    static constexpr int NW = (KP > 8) ? 2 : 1; // 32-bit words of a k-mer (16 columns each)
    // 16 < k <= 20: the second word of a k-mer holds 4 columns (one byte). The four k-mers of a quad share ONE word
    // there (byte i = columns 16..19 of k-mer i), which is counted once per quad instead of once per k-mer (C4: k = 20).
    static constexpr bool HI4 = (KP == 9 || KP == 10);
    using Word = typename std::conditional<(KP > 8), uint64_t, uint32_t>::type; // a k-mer as the gathers deliver it
    uint32_t nib[HI4 ? 1 : NW][3][2]; // [word][base - 1][column parity]: 4-bit fields, field m = column 16 word + 2 m + parity
    uint32_t byt[NW][3][2][2];        // [..][nibble parity h]: 8-bit fields, field q = column 16 word + 4 q + 2 h + parity
    uint32_t hq[HI4 ? 3 : 1];         // HI4: [base - 1] 2-bit fields of the shared word, field 4 i + c = column 16 + c of k-mer i
    int quads;                        // quads since the last nibble spill (<= 3)
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int w = 0; w < NW; ++w)
#pragma unroll
            for (int b = 0; b < 3; ++b)
#pragma unroll
                for (int p = 0; p < 2; ++p) {
                    if (!HI4 || w == 0) nib[HI4 ? 0 : w][b][p] = 0;
                    byt[w][b][p][0] = byt[w][b][p][1] = 0;
                }
        if (HI4) hq[0] = hq[1] = hq[2] = 0;
        quads = 0;
    }
    __device__ __forceinline__ void spill() {
#pragma unroll
        for (int w = 0; w < NW; ++w)
#pragma unroll
            for (int b = 0; b < 3; ++b)
#pragma unroll
                for (int p = 0; p < 2; ++p) {
                    uint32_t v;
                    if (HI4 && w == 1) {
                        v = (p == 0 ? hq[b] : (hq[b] >> 2)) & 0x33333333u; // (<= 3 per field: three quads)
                    } else {
                        v = nib[HI4 ? 0 : w][b][p];
                        nib[HI4 ? 0 : w][b][p] = 0;
                    }
                    byt[w][b][p][0] += v & 0x0F0F0F0Fu;
                    byt[w][b][p][1] += (v >> 4) & 0x0F0F0F0Fu;
                }
        if (HI4) hq[0] = hq[1] = hq[2] = 0;
        quads = 0;
    }
    // four k-mers (an invalid draw passes 0: base 0 everywhere, counted nowhere)
    __device__ __forceinline__ void add4(const Word x[4]) {
        if (quads == 3) spill();
#pragma unroll
        for (int w = 0; w < (HI4 ? 1 : NW); ++w) {
            uint32_t f[4][3];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint32_t v = (uint32_t)(x[i] >> (32 * w)), t = v >> 1;
                f[i][0] = v & ~t & 0x55555555u;
                f[i][1] = ~v & t & 0x55555555u;
                f[i][2] = v & t & 0x55555555u;
            }
#pragma unroll
            for (int b = 0; b < 3; ++b) {
                const uint32_t s3 = f[0][b] + f[1][b] + f[2][b]; // <= 3 per 2-bit field
                nib[w][b][0] += (s3 & 0x33333333u) + (f[3][b] & 0x11111111u);
                nib[w][b][1] += ((s3 >> 2) & 0x33333333u) + ((f[3][b] >> 2) & 0x11111111u);
            }
        }
        if constexpr (HI4) {
            const uint32_t h01 = __byte_perm((uint32_t)((uint64_t)x[0] >> 32), (uint32_t)((uint64_t)x[1] >> 32), 0x0040);
            const uint32_t h23 = __byte_perm((uint32_t)((uint64_t)x[2] >> 32), (uint32_t)((uint64_t)x[3] >> 32), 0x0040);
            const uint32_t v = __byte_perm(h01, h23, 0x5410), t = v >> 1; // byte i = columns 16..19 of k-mer i
            hq[0] += v & ~t & 0x55555555u;
            hq[1] += ~v & t & 0x55555555u;
            hq[2] += v & t & 0x55555555u;
        }
        ++quads;
    }
    // Warp totals into dst[j*4 + b] for b = 1, 2, 3 and columns j < k; dst[j*4] gets `added` (the k-mers the whole warp
    // added since the last flush; finish() turns it into the count of base 0). At most 252 k-mers per lane between
    // flushes. first: dst is written, else increased. Reduction number `it` (two byte fields widened to 16 bits, one
    // REDUX.SUM) is kept by lane `it`, so the results leave with two stores per lane instead of a predicated
    // read-modify-write per reduction. HI4: the byte fields of the shared word belong to k-mer slots g and g + 2 of the
    // same column 16 + 2 h + p; the lanes g = 0 / 1 of a (b, p, h) group add their halves up.
    __device__ __forceinline__ void flush(int32_t *dst, int k, int added, bool first, int lane) {
        spill();
        uint32_t mine[NW] = {};
#pragma unroll
        for (int w = 0; w < NW; ++w)
#pragma unroll
            for (int b = 0; b < 3; ++b)
#pragma unroll
                for (int p = 0; p < 2; ++p)
#pragma unroll
                    for (int h = 0; h < 2; ++h)
#pragma unroll
                        for (int g = 0; g < 2; ++g) { // g = 0: byte fields 0, 2; g = 1: byte fields 1, 3
                            const int it = (((b * 2 + p) * 2 + h) * 2 + g); // 0 .. 23 within word w
                            const int col0 = (HI4 && w == 1) ? 16 + 2 * h + p : 16 * w + 4 * g + 2 * h + p;
                            if (col0 < 2 * KP) {                            // (first column of the pair exists)
                                const uint32_t s = __reduce_add_sync(FULL, (byt[w][b][p][h] >> (8 * g)) & 0x00FF00FFu);
                                if (lane == it) mine[w] = s;
                            }
                        }
        {
            const int g = lane & 1, h = (lane >> 1) & 1, p = (lane >> 2) & 1, b = lane >> 3;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                const int32_t v0 = (int32_t)(mine[w] & 0xFFFFu), v1 = (int32_t)(mine[w] >> 16);
                if (HI4 && w == 1) {
                    const int32_t half = v0 + v1, tot = half + __shfl_xor_sync(FULL, half, 1);
                    const int c = 16 + 2 * h + p;
                    if (lane < 24 && g == 0 && c < k) dst[c * 4 + b + 1] = first ? tot : dst[c * 4 + b + 1] + tot;
                } else if (lane < 24) {
                    const int c0 = 16 * w + 4 * g + 2 * h + p, c1 = c0 + 8; // columns of the two 16-bit halves
                    if (c0 < k) dst[c0 * 4 + b + 1] = first ? v0 : dst[c0 * 4 + b + 1] + v0;
                    if (c1 < k) dst[c1 * 4 + b + 1] = first ? v1 : dst[c1 * 4 + b + 1] + v1;
                }
            }
        }
#pragma unroll
        for (int w = 0; w < NW; ++w)
#pragma unroll
            for (int b = 0; b < 3; ++b)
#pragma unroll
                for (int p = 0; p < 2; ++p) byt[w][b][p][0] = byt[w][b][p][1] = 0;
        if (lane < k) dst[lane * 4] = first ? added : dst[lane * 4] + added;
        __syncwarp();
    }
    // after the last flush: base 0 = what the other three left
    static __device__ __forceinline__ void finish(int32_t *dst, int k, int lane) {
        if (lane < k) dst[lane * 4] -= dst[lane * 4 + 1] + dst[lane * 4 + 2] + dst[lane * 4 + 3];
        __syncwarp();
    }
};

// k-mer at base `pos` of row i of a packed set, as one (k <= 16) or two 32-bit words. SROWS: the set is in shared memory.
// (__funnelshift_r shifts by its count & 31, and (2 pos) & 31 = 2 (pos & 15).)
template <int KP, bool SROWS>
__device__ __forceinline__ typename KmerCounter<KP>::Word gather_kmer(const uint32_t *__restrict__ rows, int row_words, int i, int pos) {
    uint32_t w0, w1, w2 = 0;
    if (SROWS) {
        const uint32_t *p = rows + (i * row_words + (pos >> 4));
        w0 = p[0];
        w1 = p[1];
        if (KP > 8) w2 = p[2];
    } else {
        const uint32_t *p = rows + (size_t)i * row_words + (pos >> 4);
        w0 = __ldg(p);
        w1 = __ldg(p + 1);
        if (KP > 8) w2 = __ldg(p + 2);
    }
    const uint32_t lo = __funnelshift_r(w0, w1, 2 * pos);
    if constexpr (KP > 8) {
        return ((uint64_t)__funnelshift_r(w1, w2, 2 * pos) << 32) | lo;
    } else {
        return lo;
    }
}
// the same from the gather copy (DeviceSeqs::wide), k <= 25: one 8-byte load
template <int KP>
__device__ __forceinline__ typename KmerCounter<KP>::Word gather_kmer_wide(const uint64_t *__restrict__ wide, int wide_words, int i, int pos) {
    const uint64_t v = __ldg(wide + (size_t)i * wide_words + (pos >> 3)) >> (2 * (pos & 7));
    return (typename KmerCounter<KP>::Word)v;
}

// counts over the sites of all sequences except `exclude` (sites < 0 = no site), positions shifted
// by `mode`: the fused PFM of fs:392-396 (exclude = held-out) or the all-sites total. All T warps
// of the team take part; ends with a team sync. GAP and gap != null: also the gap row, Gaps per column, into gap[32].
template <int KP, int T, bool GAP = false>
__device__ __forceinline__ void site_counts(const DeviceSeqs &s, const int32_t *sites, int exclude, int k, int mode,
                                            int32_t *total, const uint32_t *lut, int32_t *fix, int tid, int32_t *gap = nullptr) {
    constexpr int THREADS = 32 * T;
    for (int e = tid; e < MAX_COLS * 4; e += THREADS) total[e] = 0;
    if (s.mask != nullptr && tid < MAX_COLS) fix[tid] = 0;
    if (GAP && gap != nullptr && tid < MAX_COLS) gap[tid] = 0;
    team_sync<T>();
    Hist<KP> h;
    h.clear();
    const int iters = (s.n + THREADS - 1) / THREADS;
    for (int it0 = 0; it0 < iters; it0 += 255) { // byte counters hold 255 adds per thread
        const int it1 = min(iters, it0 + 255);
        for (int it = it0; it < it1; ++it) {
            const int i = it * THREADS + tid;
            h.maybe_spill(1);
            if (i < s.n && i != exclude) {
                const int site = __ldcg(sites + i);
                if (site >= 0) {
                    const int pos = shifted_site(site, __ldg(s.len + i), k, mode);
                    h.add(kmer_global<KP>(s.packed + (size_t)i * s.row_words, pos), lut);
                    if (row_masked(s, i)) {
                        if (GAP && gap != nullptr) hist_fix_gap(s.mask, s.row_words, i, pos, k, fix, gap);
                        else hist_fix(s.mask, s.row_words, i, pos, k, fix);
                    }
                }
            }
        }
        h.template flush_add<(T > 1)>(total, k, tid & 31);
    }
    team_sync<T>();
    if (s.mask != nullptr) {
        if (tid < k) total[tid * 4] -= fix[tid];
        team_sync<T>();
    }
}

// ------------------------------------------------------------------------------------------------
// PWM tables for one held-out sequence (one warp)
// ------------------------------------------------------------------------------------------------
// Leave-one-out count c = counts - own, then W(c, b) and its fixed-point log2 are gathered from the
// precomputed table (normalizePPM fs:255-261 + createPositionWeightMatrix fs:282-287 evaluated once
// per distinct count instead of once per window).
// WSMEM: wtab is a copy in shared memory (chain_cluster_kernel), else global memory read through the read-only path
template <int KP, bool MASKED, bool WSMEM = false>
__device__ __forceinline__ void build_tables_impl(const WarpTables &W, const int32_t *counts, bool has_own, uint64_t own, int k,
                                                  const WEnt *__restrict__ wtab, int lane, uint64_t own_mask) {
    constexpr int NE = (8 * KP + 31) / 32;  // passes over the (column, base) entries: entry e = lane + 32 i
    constexpr int NP = (16 * KP + 31) / 32; // passes over the pair-table entries
    int32_t lg[NE];
#pragma unroll
    for (int i = 0; i < NE; ++i) {
        const int e = lane + 32 * i;
        const int j = e >> 2, b = e & 3;
        double w = 1.0;
        lg[i] = 0;
        if (e < 8 * KP && j < k) {
            int c = counts[e];
            if (has_own && (int)((own >> (2 * j)) & 3u) == b && !(MASKED && ((own_mask >> (2 * j)) & 1u))) c -= 1; // (a masked own base was never counted)
            const int4 *ent = reinterpret_cast<const int4 *>(wtab + (size_t)c * 4 + b);
            const int4 raw = WSMEM ? *ent : __ldg(ent);
            w = __hiloint2double(raw.y, raw.x);
            lg[i] = raw.z;
        }
        if (e < 8 * KP) W.wcol[e] = w;
    }
    // pair table straight from the registers: entry (p, nib) = lg(column 2p, base nib & 3) + lg(column 2p + 1, base nib >> 2).
    // Pass t, lane l holds p = 2 t + (l >> 4), nib = l & 15; both addends sit in register lg[t >> 1] of the lanes
    // 16 (t & 1) + 8 (l >> 4) + {nib & 3, 4 + (nib >> 2)}.
    const int s0 = 8 * (lane >> 4) + (lane & 3), s1 = 8 * (lane >> 4) + 4 + ((lane >> 2) & 3);
#pragma unroll
    for (int t = 0; t < NP; ++t) {
        const int32_t v = __shfl_sync(FULL, lg[t >> 1], s0 + 16 * (t & 1)) + __shfl_sync(FULL, lg[t >> 1], s1 + 16 * (t & 1));
        const int idx = lane + 32 * t;
        if (idx < 16 * KP) W.ptab[idx] = v;
    }
    __syncwarp();
}

template <int KP>
__device__ __forceinline__ void build_tables(const WarpTables &W, const int32_t *counts, bool has_own, uint64_t own, int k,
                                             const WEnt *__restrict__ wtab, int lane) {
    build_tables_impl<KP, false>(W, counts, has_own, own, k, wtab, lane, 0);
}
// the held-out sequence's own site covers symbols outside A,C,G,T (own_mask: 0b11 at those columns); rare, out of line
template <int KP>
__device__ __noinline__ void build_tables_masked(const WarpTables &W, const int32_t *counts, uint64_t own, int k,
                                                 const WEnt *__restrict__ wtab, int lane, uint64_t own_mask) {
    build_tables_impl<KP, true>(W, counts, true, own, k, wtab, lane, own_mask);
}

// ------------------------------------------------------------------------------------------------
// exact float64 window score: Array.fold (fun (pos, v) b -> pos + 1, v * pwm.[b, pos]) (0, 1.) (fs:290-293)
// ------------------------------------------------------------------------------------------------
template <int OFF>
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1+%2];" : "=d"(v) : "r"(addr), "n"(OFF));
    return v;
}
// factor of column J: wcol[J][base J of the k-mer]; the address register is (base * 8) | table address (the table is
// 32-byte aligned: one shift + one LOP3), the immediate selects the column (32 B each)
template <int C>
__device__ __forceinline__ double column_factor(uint32_t lo, uint32_t hi, uint32_t wcol_addr) {
    const uint32_t word = C < 16 ? lo : hi;
    constexpr int sh = 2 * (C & 15); // bit position of the base code inside its word
    const uint32_t off = (sh >= 3 ? (word >> (sh - 3)) : (word << (3 - sh))) & 24u;
    return lds_f64<C * 32>(off | wcol_addr);
}
// product of the factors of columns 0 .. J - 1, left to right: (w0 * w1) * w2 ... (fs:291-292; the fold's 1 * w0 is w0)
template <int KP, int J>
struct WindowProduct {
    static __device__ __forceinline__ double upto(uint32_t lo, uint32_t hi, uint32_t wcol_addr) {
        if constexpr (J == 1) {
            return column_factor<0>(lo, hi, wcol_addr);
        } else {
            const double prev = WindowProduct<KP, J - 1>::upto(lo, hi, wcol_addr);
            return __dmul_rn(prev, column_factor<J - 1>(lo, hi, wcol_addr));
        }
    }
};

// Every window over all 2 KP columns of wcol: every table this reads holds 1.0 in the four entries of each column
// k .. 2 KP - 1 (build_tables_impl, the MotifSampler's odds and background tables), and x * 1.0 == x exactly in float64
// (device float64 keeps subnormals), so the product is the reference's k-factor fold bit for bit.
template <int KP>
__device__ __forceinline__ double exact_window(const uint32_t *row, int w, const double *wcol) {
    const uint64_t kmer = kmer_shared<KP>(row, w);
    return WindowProduct<KP, 2 * KP>::upto((uint32_t)kmer, (uint32_t)(kmer >> 32), smem_u32(wcol));
}

__device__ __forceinline__ bool better(double ohv, int ow, double hv, int w) { return ohv > hv || (ohv == hv && ow < w); }

// sum over the warp; every lane ends with it
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// (max value, lowest index) over the warp; every lane ends with the result
__device__ __forceinline__ void warp_argmax(double &hv, int &w) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double ohv = __shfl_xor_sync(FULL, hv, o);
        const int ow = __shfl_xor_sync(FULL, w, o);
        if (better(ohv, ow, hv, w)) {
            hv = ohv;
            w = ow;
        }
    }
}

// the reference loop itself (fs:302-314): every window in float64, first strict maximum from (0., 0)
template <int KP>
__device__ __forceinline__ void scan_exact_all(const uint32_t *row, int W, const double *wcol, int lane,
                                               double &hv_out, int &w_out) {
    double hv = 0.0;
    int hw = 0;
    for (int w = lane; w < W; w += 32) {
        const double p = exact_window<KP>(row, w, wcol);
        if (p > hv) {
            hv = p;
            hw = w;
        }
    }
    warp_argmax(hv, hw);
    hv_out = hv;
    w_out = hw;
}

// the same loop for a sequence with symbols outside A,C,G,T: a window that holds one scores 0 (its PWM
// row is 0, fs:283-287), every other window is scored as above
template <int KP>
__device__ __noinline__ void scan_exact_masked(const uint32_t *row, const uint32_t *__restrict__ mask, int row_words, int n,
                                               int W, int k, const double *wcol, int lane, double &hv_out, int &w_out) {
    double hv = 0.0;
    int hw = 0;
    for (int w = lane; w < W; w += 32) {
        if (mask_kmer(mask, row_words, n, w, k) != 0) continue;
        const double p = exact_window<KP>(row, w, wcol);
        if (p > hv) {
            hv = p;
            hw = w;
        }
    }
    warp_argmax(hv, hw);
    hv_out = hv;
    w_out = hw;
}

// ------------------------------------------------------------------------------------------------
// ranking pass: int32 fixed-point log2-odds, two columns per lookup
// ------------------------------------------------------------------------------------------------
// A chunk is CH consecutive windows handled by one lane. Even windows 2e use the nibbles at bit
// 4(e+p) of the chunk's aligned bit string, odd windows those at bit 4(e+p)+2, so CH/2 + KP - 1
// nibble extractions per parity serve CH/2 windows x KP lookups. Returns the chunk maximum of
// key = (sum << 8) | (255 - round), i.e. the low 8 bits identify the chunk among the lane's chunks.
// The lookups are issued as ld.shared [reg + imm]: the register is (nibble * 4) | shared address of the warp's pair
// table -- one shift and one LOP3 per nibble, which is why the per-warp tables are 64-byte aligned -- and the immediate
// selects the column pair (64 B per table).
template <int OFF>
__device__ __forceinline__ int32_t lds_ptab(uint32_t addr) {
    int32_t v;
    asm volatile("ld.shared.s32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
}
template <int KP, int P>
struct PairSum { // sum over column pairs P .. KP-1 of ptab[p][nibble e + p]
    static __device__ __forceinline__ int32_t of(const uint32_t *ad, int e) {
        return lds_ptab<P * 64>(ad[e + P]) + PairSum<KP, P + 1>::of(ad, e);
    }
};
template <int KP>
struct PairSum<KP, KP> {
    static __device__ __forceinline__ int32_t of(const uint32_t *, int) { return 0; }
};

template <int KP, int CH, bool MASK>
__device__ __forceinline__ int32_t score_chunk(const uint32_t *a, const uint32_t *b, uint32_t ptab_addr, int idx, int lim) {
    constexpr int NE = CH / 2 + KP - 1;
    uint32_t adE[NE], adO[NE]; // (nibble << 2) | table address, even / odd windows
#pragma unroll
    for (int t = 0; t < NE; ++t) {
        const int j = t & 7;
        const uint32_t xe = a[t >> 3], xo = b[t >> 3];
        adE[t] = ((j == 0 ? (xe << 2) : (xe >> (4 * j - 2))) & 0x3cu) | ptab_addr;
        adO[t] = ((j == 0 ? (xo << 2) : (xo >> (4 * j - 2))) & 0x3cu) | ptab_addr;
    }
    int32_t key[CH];
#pragma unroll
    for (int i = 0; i < CH; ++i) {
        const int e = i >> 1;
        int32_t v = idx + ((i & 1) ? PairSum<KP, 0>::of(adO, e) : PairSum<KP, 0>::of(adE, e));
        if (MASK) v = (i < lim) ? v : INT32_MIN;
        key[i] = v;
    }
#pragma unroll
    for (int st = 1; st < CH; st *= 2) // max tree (the compiler fuses pairs into 3-input VIMNMX3)
#pragma unroll
        for (int i = 0; i + st < CH; i += 2 * st) key[i] = max(key[i], key[i + st]);
    return key[0];
}

template <int KP, int CH>
struct ScanGeom {
    static constexpr int NB = CH + 2 * KP - 1;  // bases a chunk touches
    static constexpr int NWA = (NB + 15) / 16;  // aligned words
    static constexpr int RPS = 256;             // rounds per segment (round index fits 8 bits)
    static constexpr int CPS = 32 * RPS;        // chunks per segment
};

// first window of chunk c: the last chunk is pulled back so that every chunk is full (its overlap
// with the previous chunk only rescans windows, harmless for a maximum); rows shorter than one
// chunk (W < CH) are the single masked case
template <int CH>
__device__ __forceinline__ int chunk_base(int c, int W) { return max(0, min(c * CH, W - CH)); }

// per-lane best chunk key M1 (from segment S1), best key among the lane's OTHER chunks M2
template <int KP, int CH>
__device__ __forceinline__ void scan_fast(const uint32_t *row, int W, const int32_t *ptab, int lane, int32_t &M1,
                                          int32_t &M2, int &S1) {
    using G = ScanGeom<KP, CH>;
    const int n_chunks = (W + CH - 1) / CH;
    const uint32_t ptab_addr = smem_u32(ptab); // 64-byte aligned (checked once per kernel: tables_aligned)
    M1 = INT32_MIN;
    M2 = INT32_MIN;
    S1 = 0;
    for (int seg = 0, c0 = 0; c0 < n_chunks; ++seg, c0 += G::CPS) {
        const int c_end = min(n_chunks, c0 + G::CPS);
        int idx = 255;
        for (int c = c0 + lane; c < c_end; c += 32, --idx) {
            const int base0 = chunk_base<CH>(c, W);
            const uint32_t *p = row + (base0 >> 4);
            const int sh = (base0 & 15) * 2;
            uint32_t raw[G::NWA + 1], a[G::NWA + 1], b[G::NWA];
#pragma unroll
            for (int i = 0; i <= G::NWA; ++i) raw[i] = p[i];
#pragma unroll
            for (int i = 0; i < G::NWA; ++i) a[i] = __funnelshift_r(raw[i], raw[i + 1], sh);
            a[G::NWA] = 0;
#pragma unroll
            for (int i = 0; i < G::NWA; ++i) b[i] = __funnelshift_r(a[i], a[i + 1], 2);
            int32_t cm;
            if (W >= CH) cm = score_chunk<KP, CH, false>(a, b, ptab_addr, idx, CH); // warp-uniform branch
            else cm = score_chunk<KP, CH, true>(a, b, ptab_addr, idx, W);
            if (cm > M1) {
                M2 = max(M2, M1);
                M1 = cm;
                S1 = seg;
            } else {
                M2 = max(M2, cm);
            }
        }
    }
}

// getBestPWMSsWithBPV (fs:301-314) for the staged row: (raw float64 maximum, first argmax).
// Returns true when the all-windows float64 path has to be taken.
template <int KP, int CH>
__device__ __forceinline__ bool pick_argmax_ch(const WarpTables &T, const uint32_t *row, int W, int k, int lane,
                                               double &hv_out, int &w_out) {
    using G = ScanGeom<KP, CH>;
    int32_t M1, M2;
    int S1;
    scan_fast<KP, CH>(row, W, T.ptab, lane, M1, M2, S1);
    const int32_t M = __reduce_max_sync(FULL, M1);
    // |key/256 - true log2 score * 2^11| <= k/2 units for every window, so any window whose exact
    // product can reach the maximum lies in a chunk whose key >= M - (k + 1) units (index bits: 255 more)
    const int32_t thr = M - (((k + 1) << KEY_IDX_BITS) + 255);
    if (__ballot_sync(FULL, M2 >= thr)) return true; // a lane with two candidate chunks: rescan exactly
    unsigned cand = __ballot_sync(FULL, M1 >= thr);
    // every window of every candidate chunk is re-scored in float64, one window per lane
    const bool single = (cand & (cand - 1)) == 0;
    double p = 0.0;
    int w = INT32_MAX;
    while (cand) {
        const int src = __ffs(cand) - 1;
        cand &= cand - 1;
        const int32_t key = __shfl_sync(FULL, M1, src);
        const int seg = __shfl_sync(FULL, S1, src);
        const int base0 = chunk_base<CH>(seg * G::CPS + src + 32 * (255 - (key & 255)), W);
        const int wi = base0 + lane;
        if (lane < CH && wi < W) {
            const double pi = exact_window<KP>(row, wi, T.wcol);
            if (better(pi, wi, p, w)) {
                p = pi;
                w = wi;
            }
        }
    }
    if (single) { // lanes hold ascending windows: the first lane with the largest product is the first maximum
        const uint32_t hi = (uint32_t)__double2hiint(p), mh = __reduce_max_sync(FULL, hi);
        const uint32_t lo = (hi == mh) ? (uint32_t)__double2loint(p) : 0u, ml = __reduce_max_sync(FULL, lo);
        const int src = __ffs(__ballot_sync(FULL, hi == mh && lo == ml)) - 1;
        p = __shfl_sync(FULL, p, src);
        w = __shfl_sync(FULL, w, src);
    } else {
        warp_argmax(p, w);
    }
    hv_out = p;
    w_out = w;
    return false;
}

// masked_seq >= 0: the held-out sequence holds symbols outside A,C,G,T (s.mask != null)
template <int KP>
__device__ __forceinline__ bool pick_argmax(const WarpTables &T, const uint32_t *row, int W, int k, int fast_ok, int lane,
                                            double &hv_out, int &w_out, const DeviceSeqs *s = nullptr, int masked_seq = -1) {
    if (masked_seq >= 0) {
        scan_exact_masked<KP>(row, s->mask, s->row_words, masked_seq, W, k, T.wcol, lane, hv_out, w_out);
        return true;
    }
    bool slow = !fast_ok;
    if (!slow) {
        if (W > 256) slow = pick_argmax_ch<KP, 16>(T, row, W, k, lane, hv_out, w_out);
        else if (W > 128) slow = pick_argmax_ch<KP, 8>(T, row, W, k, lane, hv_out, w_out);
        else slow = pick_argmax_ch<KP, 4>(T, row, W, k, lane, hv_out, w_out);
    }
    if (slow) scan_exact_all<KP>(row, W, T.wcol, lane, hv_out, w_out);
    return slow;
}

__device__ __forceinline__ double log2_ref(double x) { return log(x) / LN2; } // fs:303 via FSharpAux

// `if fst tmp > fst acc.[n]` (fs:402) on log2 scores, decided from the raw products whenever the
// two logs cannot collide
// hv_old = NaN marks a caller-supplied start state: only its log2 score (score_old) is known.
__device__ __forceinline__ bool score_improves(double hv_new, double hv_old, double score_old) {
    if (hv_old != hv_old) return log2_ref(hv_new) > score_old;
    if (!(hv_new > hv_old)) return false;
    if (hv_new * (1.0 - 0x1p-30) > hv_old) return true;
    return log2_ref(hv_new) > log2_ref(hv_old);
}

} // namespace gibbs
