// gibbssampling_b200/csrc/gibbs_batch_tu.cu -- one group of chain_batch_kernel instantiations per translation unit.
// Compiled several times by _build.py (BATCH_GROUPS) with -DGIBBS_TU_NAME=launch_batch_xxx -DGIBBS_TU_T=<warps per chain>
// -DGIBBS_TU_MASKED=0|1 -DGIBBS_TU_DRIFT=0|1 [-DGIBBS_TU_INIT_ONLY=1], each time for the 16 k-widths. Units of their own,
// so that the chain_kernel units keep their code generation (see gibbs_chain_tu.cu).
#include "gibbs_batch.cuh"

#ifndef GIBBS_TU_INIT_ONLY
#define GIBBS_TU_INIT_ONLY 0
#endif
#if !defined(GIBBS_TU_NAME) || !defined(GIBBS_TU_T) || !defined(GIBBS_TU_MASKED) || !defined(GIBBS_TU_DRIFT)
#error "compile with -DGIBBS_TU_NAME=... -DGIBBS_TU_T=... -DGIBBS_TU_MASKED=... -DGIBBS_TU_DRIFT=... (see _build.py)"
#endif

namespace gibbs {

template <int KPV>
static cudaError_t launch_one(const ChainArgs &run, const BatchTable &bt, int grid, int smem, cudaStream_t stream) {
    auto kernel = chain_batch_kernel<KPV, GIBBS_TU_T, GIBBS_TU_MASKED != 0, GIBBS_TU_DRIFT != 0, GIBBS_TU_INIT_ONLY != 0>;
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
    }
    kernel<<<grid, 32 * GIBBS_TU_T, smem, stream>>>(run, bt);
    return cudaGetLastError();
}

// smem = team_smem_bytes(row_words, GIBBS_TU_T) (dynamic; the set's ChainArgs copy is static shared memory)
cudaError_t GIBBS_TU_NAME(const ChainArgs &run, const BatchTable &bt, int grid, int smem, cudaStream_t stream) {
    switch ((run.k + 1) / 2) {
#define X(KPV) case KPV: return launch_one<KPV>(run, bt, grid, smem, stream);
        X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16)
#undef X
    default: return cudaErrorInvalidValue;
    }
}

} // namespace gibbs
