// inst_run.cu -- one translation unit per (real type, est_bias, direct_orien_method, multirate_ekf); compiled
// with -DQ_T=double|float -DQ_BIAS=0|1 -DQ_DIRECT=0|1 -DQ_MR=0|1.  Holds the explicit-stream and the
// synthetic-noise instantiations of the fused multi-tick kernel, with and without per-filter parameters.
#include "launch.hpp"

namespace qekf {

template <typename T, bool BIAS, bool DIRECT, bool SYNTH, bool MR, bool PF, bool STATS>
cudaError_t launch_run(const RunArgs<T> &a, unsigned grid, size_t smem, cudaStream_t stream)
{
    auto kern = run_kernel<T, BIAS, DIRECT, SYNTH, MR, PF, BlockOf<T>::value, STATS>;
    cudaError_t e = prep_kernel(kern, smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, BlockOf<T>::value, smem, stream>>>(a);
    return cudaGetLastError();
}

template <typename T, bool BIAS, bool DIRECT, bool MR>
cudaError_t launch_tick(const RunArgs<T> &a, const double *pose8, int tag_mode, double *out, int n_out, cudaStream_t stream)
{
    constexpr int N = BIAS ? 15 : 9;
    auto kern = tick_kernel<T, BIAS, DIRECT, MR>;
    const size_t smem = (size_t)TICK_BLOCK * (N * (N + 1) / 2) * sizeof(T) + VOTE_WORDS * sizeof(int) +
                        (size_t)TICK_BLOCK * (MR ? MR_SCRATCH_INTS : SR_SCRATCH_INTS) * sizeof(int32_t);
    static unsigned prepared = 0;          // per instantiation and device: the attribute call is not free on a 200 Hz path
    int dev = 0;
    cudaGetDevice(&dev);
    if (!(prepared & (1u << (dev & 31)))) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        prepared |= 1u << (dev & 31);
    }
    const unsigned grid = (unsigned)((a.st.n + TICK_BLOCK - 1) / TICK_BLOCK);
    kern<<<grid, TICK_BLOCK, smem, stream>>>(a, pose8, tag_mode, out, n_out);
    return cudaGetLastError();
}
template cudaError_t launch_tick<Q_T, (Q_BIAS != 0), (Q_DIRECT != 0), (Q_MR != 0)>(const RunArgs<Q_T> &, const double *, int,
                                                                                   double *, int, cudaStream_t);

#define INST(S, PF_, ST)                                                                                              \
    template cudaError_t launch_run<Q_T, (Q_BIAS != 0), (Q_DIRECT != 0), S, (Q_MR != 0), PF_, ST>(const RunArgs<Q_T> &, \
                                                                                                   unsigned, size_t,      \
                                                                                                   cudaStream_t);
INST(false, false, false)
INST(true, false, true)
INST(false, true, false)
INST(true, true, true)
INST(false, false, true)      // explicit streams scored against per-filter truth (qekf_run_with_truth)
INST(false, true, true)

}  // namespace qekf
