// gibbssampling_b200/csrc/gibbs_cluster.cuh -- the last stages of the straggler hand-over: ONE chain on a thread-block
// cluster of C CTAs x 16 warps (sm_100a only).
//
// A run ends with a handful of chains that need many more sweeps than the rest (13 to 35+ at C2). A 16-warp team is
// issue-bound on its own SM (16 site updates per ~3.7 us round), so with fewer chains than SMs left the only way to
// shorten the tail is to give one chain several SMs. The C CTAs of a cluster work as one team of C x 16 warps: a round
// scores C x 16 consecutive held-out sequences, every warp publishes its outcome into the shared memory of all C CTAs
// (st.shared::cluster, DSMEM), one cluster barrier closes the round, and every CTA then takes the same decisions from
// its own copy of the flags -- the commit rule is chain_kernel's: results commit in order up to and including the first
// warp whose accepted update moves a site; the rest of the round is redone. Each CTA keeps its own copy of the all-sites
// counts and applies the mover's -old / +new k-mer itself, so nothing but flags and two k-mers ever crosses SMs.
// The committed sequence of site updates is exactly the reference's sequential sweep (fs:381-408, fs:350-377,
// fs:318-346), whatever C is.
//
// Fixed background, A,C,G,T-only sets, ranking pass usable (the benchmarked family). The PWM value table W(c, b) sits in
// shared memory (one CTA per SM: the space is free), rows are prefetched per warp with cp.async for the round that
// follows when nothing moves.
#pragma once
#include "gibbs_kernels.cuh"

namespace gibbs {

constexpr int CL_T = 16; // warps per CTA

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(const void *smem_ptr, uint32_t rank) {
    uint32_t out;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(out) : "r"(smem_u32(smem_ptr)), "r"(rank));
    return out;
}
__device__ __forceinline__ void st_cluster_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void st_cluster_u64(uint32_t addr, uint64_t v) {
    asm volatile("st.shared::cluster.u64 [%0], %1;" ::"r"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory"); }

// shared memory of one CTA
//   [0, 512)            total: counts over all current sites (own copy per CTA)
//   [512, 640)          fix (unused: sets with masked symbols never get here) / scratch
//   [640, 704)          lut of the histogram (site_counts)
//   [704, 704 + 8 GW)   flags [2][GW]
//   then                delta [2][GW][2] uint64: (old k-mer, new k-mer) of a mover
//   then 16 B           control word written by rank 0 (pause decision)
//   then                per-warp tables 16 x WARP_TABLE_BYTES
//   then                per-warp rows 16 x 2 x row_words x 4
//   then                wtab copy n x 4 x 16 B
template <int C>
__host__ __device__ constexpr int cl_flags_off() { return 704; }
template <int C>
__host__ __device__ constexpr int cl_delta_off() { return cl_flags_off<C>() + 2 * C * CL_T * 4; }
template <int C>
__host__ __device__ constexpr int cl_ctl_off() { return cl_delta_off<C>() + 2 * C * CL_T * 16; }
template <int C>
__host__ __device__ constexpr int cl_tables_off() { return (cl_ctl_off<C>() + 16 + 63) / 64 * 64; }
template <int C>
__host__ __device__ inline size_t cluster_smem_bytes(int n, int row_words) {
    return (size_t)cl_tables_off<C>() + (size_t)CL_T * WARP_TABLE_BYTES + (size_t)CL_T * 2 * row_words * 4 + (size_t)n * 4 * sizeof(WEnt);
}

template <int KP, int C>
static __global__ void __launch_bounds__(32 * CL_T, 1) chain_cluster_kernel(const ChainArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int T = CL_T, THREADS = 32 * CL_T, GW = C * CL_T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t crank = cluster_ctarank();
    const int gw = (int)crank * T + warp; // position of this warp in the team of GW warps
    const int entry = blockIdx.x / C;     // one cluster per list entry
    if (entry >= *a.pending_in_n) return; // (uniform over the cluster)
    const int chain = a.pending_in[entry];

    const int N = a.s.n, k = a.k, row_words = a.s.row_words;
    int32_t *total = reinterpret_cast<int32_t *>(smem_raw);
    int32_t *fix = reinterpret_cast<int32_t *>(smem_raw + 512);
    uint32_t *lut = reinterpret_cast<uint32_t *>(smem_raw + 640);
    int32_t *flags = reinterpret_cast<int32_t *>(smem_raw + cl_flags_off<C>());
    uint64_t *delta = reinterpret_cast<uint64_t *>(smem_raw + cl_delta_off<C>());
    int32_t *ctl = reinterpret_cast<int32_t *>(smem_raw + cl_ctl_off<C>());
    WarpTables WT;
    {
        unsigned char *b = smem_raw + cl_tables_off<C>() + warp * WARP_TABLE_BYTES;
        WT.wcol = reinterpret_cast<double *>(b);
        WT.ptab = reinterpret_cast<int32_t *>(b + 1024);
        WT.lgcol = reinterpret_cast<int32_t *>(b + 2048);
        WT.counts = reinterpret_cast<int32_t *>(b + 2560);
    }
    require_aligned_tables(WT);
    uint32_t *rows = reinterpret_cast<uint32_t *>(smem_raw + cl_tables_off<C>() + T * WARP_TABLE_BYTES) + warp * 2 * row_words;
    WEnt *wtab_s = reinterpret_cast<WEnt *>(smem_raw + cl_tables_off<C>() + T * WARP_TABLE_BYTES + (size_t)T * 2 * row_words * 4);

    int32_t *sites = a.sites + (size_t)chain * N;
    double *hv = a.hv + (size_t)chain * N;
    double *scores = a.scores + (size_t)chain * N;

    if (tid < 16) lut[tid] = hist_lut_entry(tid);
    {   // W(c, b) for every count: 16 B entries
        const int4 *src = reinterpret_cast<const int4 *>(a.wtab);
        int4 *dst = reinterpret_cast<int4 *>(wtab_s);
        for (int i = tid; i < N * 4; i += THREADS) dst[i] = __ldg(src + i);
    }
    // remote addresses of this warp's flag / delta slots in every CTA of the cluster (parity 0; parity 1 = + GW entries)
    uint32_t r_flag = 0, r_delta = 0;
    if (lane < C) {
        r_flag = map_to_rank(flags + gw, (uint32_t)lane);
        r_delta = map_to_rank(delta + 2 * gw, (uint32_t)lane);
    }
    __syncthreads();
    cluster_barrier(); // every CTA of the cluster is running (remote shared memory may be written from here on)

    // site_updates and window_scores per sweep, as in chain_kernel; this warp's exact rescans and discarded updates of the
    // current sweep (at most N each) are added at its end
    unsigned st_slow = 0, st_spec = 0;
    int st_sweeps = 0, capped = 0;
    int phase, sweeps_in_phase;
    {
        const int r = a.resume[chain]; // phase | capped so far << 7 | sweeps in phase << 8
        phase = r & 127;
        capped = (r >> 7) & 1;
        sweeps_in_phase = r >> 8;
    }
    bool resumed = true, paused = false;
    const int ulen = a.s.uniform_len;

    // row of sequence `seq` into slot `slot` of this warp (cp.async, 16 B per lane)
    auto fetch_row = [&](int seq, int slot) {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.s.packed + (size_t)seq * row_words);
        uint4 *dst = reinterpret_cast<uint4 *>(rows + slot * row_words);
        for (int i = lane; i < (row_words >> 2); i += 32) cp_async16(dst + i, src + i);
    };

    while (phase != PH_DONE) {
        const int mode = phase == PH_LEFT ? SHIFT_LEFT : phase == PH_RIGHT ? SHIFT_RIGHT : SHIFT_NONE;
        // all-sites counts, in every CTA: once when the greedy phase starts or resumes (then kept incrementally),
        // once per sweep for the shift phases (they read the shifted snapshot, fs:357)
        if (phase == PH_LEFT || phase == PH_RIGHT || (phase == PH_GREEDY && (sweeps_in_phase == 0 || resumed)))
            site_counts<KP, T>(a.s, sites, -1, k, mode, total, lut, fix, tid);
        resumed = false;
        bool changed = false;
        int n0 = 0;
        int width = (phase == PH_GREEDY) ? max(1, min(GW, a.min_width)) : GW;
        unsigned round = 0;
        int have = -1, have_slot = 0; // sequence whose row sits (or is arriving) in slot have_slot; the other slot is free
        // state of the sequence this warp will probably score next, prefetched into registers
        int pf_n = -1, pf_site = 0, pf_len = 0;
        double pf_hv = 0.0;
        {
            const int n = n0 + gw;
            if (n < N) {
                fetch_row(n, 0);
                have = n;
                have_slot = 0;
                pf_n = n;
                pf_site = __ldcg(sites + n);
                pf_hv = __ldcg(hv + n);
                pf_len = ulen > 0 ? ulen : __ldg(a.s.len + n);
            }
        }
        while (n0 < N) {
            const int n = n0 + gw;
            const bool active = n < N && gw < width;
            int flag = 0, w = 0, Wn = 0;
            double p = 0.0;
            uint64_t own = 0, neu = 0;
            // the row this warp needs if the round commits in full: requested now, lands while the round computes
            const int n_pred = n + GW;
            if (n < N) {
                if (have != n) { // (a partial commit moved the window: the prefetch was for another sequence)
                    cp_async_wait_all();
                    __syncwarp();
                    fetch_row(n, have_slot);
                    have = n;
                }
                cp_async_wait_all();
                __syncwarp();
            }
            const int cur_slot = have_slot;
            int nx_site = 0, nx_len = 0;
            double nx_hv = 0.0;
            if (n_pred < N) {
                fetch_row(n_pred, cur_slot ^ 1);
                nx_site = __ldcg(sites + n_pred);
                nx_hv = __ldcg(hv + n_pred);
                nx_len = ulen > 0 ? ulen : __ldg(a.s.len + n_pred);
            }
            int site_n = 0;
            if (active) {
                const uint32_t *row = rows + cur_slot * row_words;
                int len_n;
                double hv_n;
                if (pf_n == n) {
                    site_n = pf_site;
                    hv_n = pf_hv;
                    len_n = pf_len;
                } else {
                    site_n = __ldcg(sites + n);
                    hv_n = __ldcg(hv + n);
                    len_n = ulen > 0 ? ulen : __ldg(a.s.len + n);
                }
                Wn = len_n - k + 1;
                own = kmer_shared<KP>(row, shifted_site(site_n, len_n, k, mode));
                build_tables_impl<KP, false, true>(WT, total, true, own, k, wtab_s, lane, 0);
                const bool slow = pick_argmax<KP>(WT, row, Wn, k, a.fast_ok, lane, p, w);
                const bool accept = score_improves(p, hv_n, hv_n != hv_n ? __ldcg(scores + n) : 0.0); // fs:402
                const bool moved = accept && (w != site_n);
                if (moved && phase == PH_GREEDY) neu = kmer_shared<KP>(row, w);
                flag = (accept ? 1 : 0) | (moved ? 2 : 0) | (slow ? 4 : 0) | 8; // bit 3: the slot was written this round
            }
            // publish the outcome in every CTA of the cluster (lane r writes into CTA r)
            const uint32_t par = (round & 1u);
            ++round;
            if (lane < C) {
                if ((flag & 2) && phase == PH_GREEDY) {
                    st_cluster_u64(r_delta + par * GW * 16, own);
                    st_cluster_u64(r_delta + par * GW * 16 + 8, neu);
                }
                st_cluster_u32(r_flag + par * GW * 4, (uint32_t)flag);
            }
            cluster_barrier();
            // every CTA reads the same GW flags and takes the same decisions
            const int32_t *fl = flags + par * GW;
            unsigned movers_lo = __ballot_sync(FULL, lane < GW && (fl[lane < GW ? lane : 0] & 2) != 0);
            unsigned movers_hi[(GW + 31) / 32] = {};
            movers_hi[0] = movers_lo;
#pragma unroll
            for (int q = 1; q < (GW + 31) / 32; ++q) movers_hi[q] = __ballot_sync(FULL, (fl[q * 32 + lane] & 2) != 0);
            int first_mover = GW;
            bool any_moved = false;
#pragma unroll
            for (int q = (GW + 31) / 32 - 1; q >= 0; --q)
                if (movers_hi[q]) {
                    any_moved = true;
                    first_mover = q * 32 + __ffs(movers_hi[q]) - 1;
                }
            if (phase != PH_GREEDY) first_mover = GW; // shift sweeps read a snapshot: everything commits
            const int last_commit = min(first_mover, width - 1);
            changed |= any_moved;
            if (active) {
                if (gw <= last_commit) {
                    st_slow += (flag & 4) ? 1 : 0;
                    if ((flag & 1) && lane == 0) {
                        sites[n] = w;
                        hv[n] = p;
                    }
                } else {
                    st_spec += 1;
                }
            }
            const int committed = min(last_commit + 1, N - n0);
            n0 += committed;
            if (phase == PH_GREEDY) {
                if (first_mover < GW) { // in-place sweep: later n see the new site (fs:388): -old k-mer, +new k-mer
                    if (warp == 0 && lane < k) {
                        const uint64_t o = delta[(par * GW + first_mover) * 2], nw = delta[(par * GW + first_mover) * 2 + 1];
                        const int bo = (int)((o >> (2 * lane)) & 3u), bn = (int)((nw >> (2 * lane)) & 3u);
                        if (bo != bn) {
                            total[lane * 4 + bo] -= 1;
                            total[lane * 4 + bn] += 1;
                        }
                    }
                    __syncthreads(); // counts updated before the next round builds its tables
                    width = max(max(1, min(GW, a.min_width)), width >> 1);
                } else {
                    width = min(GW, width * 2);
                }
            }
            // what the prefetch holds now
            if (n_pred < N) {
                if (committed == GW) { // the prediction holds: the other slot becomes the current one
                    have = n_pred;
                    have_slot = cur_slot ^ 1;
                    pf_n = n_pred;
                    pf_site = nx_site;
                    pf_hv = nx_hv;
                    pf_len = nx_len;
                } else { // this warp's next sequence is n0 + gw: refetched at the top of the next round
                    have = -2;
                    have_slot = cur_slot;
                    pf_n = -1;
                }
            } else {
                have = -2;
                have_slot = cur_slot;
                pf_n = -1;
            }
        }
        cp_async_wait_all(); // (a prefetch past the last round may still be in flight)
        __syncwarp();
        st_sweeps += 1;
        if (lane == 0) {
            if (st_slow) atomicAdd(a.stats + ST_EXACT_RESCANS, (unsigned long long)st_slow);
            if (st_spec) atomicAdd(a.stats + ST_SPECULATED, (unsigned long long)st_spec);
        }
        st_slow = st_spec = 0;
        ++sweeps_in_phase;
        bool next = !changed; // positions(acc) = positions(bestMotif), fs:384
        if (!next && sweeps_in_phase >= a.max_sweeps) {
            next = true;
            capped = 1;
        }
        if (next) {
            sweeps_in_phase = 0;
            phase = next_phase(phase + 1, a.phase_mask);
        }
        // sweep boundary: every CTA's writes of this sweep become visible to the others (site_counts / block state of the
        // next sweep read them); rank 0 decides about a hand-over to the next stage and tells the others
        int want_pause = 0;
        if (phase != PH_DONE && a.pause_below > 0 && crank == 0 && tid == 0)
            want_pause = (*(volatile int32_t *)a.active <= a.pause_below) ? 1 : 0;
        if (crank == 0 && tid < C) st_cluster_u32(map_to_rank(ctl, (uint32_t)tid), (uint32_t)__shfl_sync((1u << C) - 1u, want_pause, 0));
        cluster_barrier();
        if (ctl[0]) {
            paused = true;
            break;
        }
    }
    cluster_barrier(); // nobody leaves while a neighbour may still write into its shared memory
    if (crank != 0) return;
    if (st_sweeps > 0) { // windows per sweep: the sum of len_n - k + 1 over the sequences, added per warp of rank 0
        unsigned long long sum_w = 0;
        for (int n = tid; n < N; n += THREADS) sum_w += (unsigned long long)(__ldg(a.s.len + n) - k + 1);
        sum_w = warp_sum_u64(sum_w);
        if (lane == 0) atomicAdd(a.stats + ST_WINDOW_SCORES, sum_w * (unsigned long long)st_sweeps);
    }
    if (tid == 0) {
        atomicAdd(a.stats + ST_SITE_UPDATES, (unsigned long long)N * (unsigned long long)st_sweeps);
        atomicAdd(a.stats + ST_SWEEPS, (unsigned long long)st_sweeps);
        if (!paused) atomicAdd(a.stats + ST_CAPPED, (unsigned long long)capped); // (a chain counts once, where it ends)
    }
    if (paused) {
        if (tid == 0) {
            a.resume[chain] = phase | (capped << 7) | (sweeps_in_phase << 8);
            a.pending_out[atomicAdd(a.pending_out_n, 1)] = chain;
        }
        return;
    }
    // (log2 highValue, highIndex), fs:303
    for (int n = tid; n < N; n += THREADS) {
        const double v = __ldcg(hv + n);
        if (v == v) scores[n] = log2_ref(v); // NaN = untouched caller-supplied entry keeps its score
    }
    __syncthreads();
    if (tid == 0) {
        double sum = 0.0; // Array.sum, left to right (fs:445)
        for (int n = 0; n < N; ++n) sum = __dadd_rn(sum, __ldcg(scores + n));
        a.sums[chain] = sum;
        if (a.active) atomicSub(a.active, 1);
    }
}

} // namespace gibbs
