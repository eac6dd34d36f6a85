// inst_step.cu -- the per-tick step kernel of qekf_step (step_kernel in ekf_kernels.cuh); one translation unit per
// (real type, est_bias, direct_orien_method, multirate_ekf), compiled with -DQ_T -DQ_BIAS -DQ_DIRECT -DQ_MR as
// inst_run.cu, with and without per-filter parameters, for every CTA size of STEP_BLOCKS.
#include "launch.hpp"

namespace qekf {

template <typename T, bool BIAS, bool DIRECT, bool MR, bool PF, int BLOCK>
static cudaError_t step_one(const StepArgs<T> *a, cudaStream_t stream)
{
    constexpr int N = BIAS ? 15 : 9;
    constexpr size_t smem = (size_t)BLOCK * (N * (N + 1) / 2) * sizeof(T);
    auto kern = step_kernel<T, BIAS, DIRECT, MR, PF, BLOCK>;
    if (!a) return prep_kernel(kern, smem);
    const unsigned grid = (unsigned)((a->st.n + BLOCK - 1) / BLOCK);
    kern<<<grid, BLOCK, smem, stream>>>(*a);
    return cudaGetLastError();
}

// a == nullptr: set the kernel's attributes only
template <typename T, bool BIAS, bool DIRECT, bool MR, bool PF>
static cudaError_t step_block(const StepArgs<T> *a, int block, cudaStream_t stream)
{
    switch (block) {
    case 32: return step_one<T, BIAS, DIRECT, MR, PF, 32>(a, stream);
    case 64: return step_one<T, BIAS, DIRECT, MR, PF, 64>(a, stream);
    case 128: return step_one<T, BIAS, DIRECT, MR, PF, 128>(a, stream);
    default: return cudaErrorInvalidValue;
    }
}

template <typename T, bool BIAS, bool DIRECT, bool MR, bool PF> cudaError_t prep_step(int block)
{
    return step_block<T, BIAS, DIRECT, MR, PF>(nullptr, block, nullptr);
}

template <typename T, bool BIAS, bool DIRECT, bool MR, bool PF>
cudaError_t launch_step(const StepArgs<T> &a, int block, cudaStream_t stream)
{
    return step_block<T, BIAS, DIRECT, MR, PF>(&a, block, stream);
}

#define INST(PF_)                                                                                                      \
    template cudaError_t prep_step<Q_T, (Q_BIAS != 0), (Q_DIRECT != 0), (Q_MR != 0), PF_>(int);                       \
    template cudaError_t launch_step<Q_T, (Q_BIAS != 0), (Q_DIRECT != 0), (Q_MR != 0), PF_>(const StepArgs<Q_T> &, int, \
                                                                                             cudaStream_t);
INST(false)
INST(true)

}  // namespace qekf
