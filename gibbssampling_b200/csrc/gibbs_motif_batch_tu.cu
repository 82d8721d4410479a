// gibbssampling_b200/csrc/gibbs_motif_batch_tu.cu -- one group of MotifSampler batch instantiations per translation unit.
// Compiled several times by _build.py (MOTIF_BATCH_GROUPS) with -DGIBBS_TU_NAME=launch_motif[2]_batch_xxx -DGIBBS_TU_M=1|2
// -DGIBBS_TU_T=<warps per restart> -DGIBBS_TU_MASKED=0|1, each time for the 16 k-widths: motif_batch_kernel<KP, T, MASKED>
// for motifAmount = 1, motif2_batch_kernel<KP> (one warp, A,C,G,T only) for motifAmount = 2. Units of their own, so that
// the motif_kernel, motif2_kernel and chain_batch_kernel units keep their code generation.
#include "gibbs_motif_batch.cuh"

#if !defined(GIBBS_TU_NAME) || !defined(GIBBS_TU_M) || !defined(GIBBS_TU_T) || !defined(GIBBS_TU_MASKED)
#error "compile with -DGIBBS_TU_NAME=... -DGIBBS_TU_M=... -DGIBBS_TU_T=... -DGIBBS_TU_MASKED=... (see _build.py)"
#endif
#if GIBBS_TU_M == 2 && (GIBBS_TU_T != 1 || GIBBS_TU_MASKED != 0)
#error "motif2_batch_kernel runs one warp per restart on A,C,G,T-only sets"
#endif

namespace gibbs {

template <int KPV>
static cudaError_t launch_one(const MotifArgs &run, const MotifBatchTable &bt, int grid, int smem, cudaStream_t stream) {
#if GIBBS_TU_M == 2
    auto kernel = motif2_batch_kernel<KPV>;
#else
    auto kernel = motif_batch_kernel<KPV, GIBBS_TU_T, GIBBS_TU_MASKED != 0>;
#endif
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    kernel<<<grid, 32 * GIBBS_TU_T, smem, stream>>>(run, bt);
    return cudaGetLastError();
}

// smem = team_smem_bytes(row_words, GIBBS_TU_T) (dynamic; the set's arguments are static shared memory)
cudaError_t GIBBS_TU_NAME(const MotifArgs &run, const MotifBatchTable &bt, int grid, int smem, cudaStream_t stream) {
    switch ((run.c.k + 1) / 2) {
#define X(KPV) case KPV: return launch_one<KPV>(run, bt, grid, smem, stream);
        X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16)
#undef X
    default: return cudaErrorInvalidValue;
    }
}

} // namespace gibbs
