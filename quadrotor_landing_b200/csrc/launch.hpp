// launch.hpp -- host-callable launchers, explicitly instantiated in inst_run.cu / inst_misc.cu so that the
// heavy kernel templates compile in parallel translation units.
#pragma once

#include <cuda_runtime.h>

#include "ekf_kernels.cuh"

namespace qekf {

// One CTA per SM.  FP64: 7 warps x 30 KB of covariance fill the shared memory.  FP32: shared memory would hold 14
// warps, but the register file decides: 12 warps at 168 registers beat 14 at 128 by 17 % (and 8 at 255, which
// does not spill at all, is as fast as 12); one lockstep CTA rather than two independent 224-thread ones, which
// drift apart and thrash the instruction cache (no_instruction 1.0 per issue in profiles/r1_13_fp32.md).
#ifdef QEKF_EXP8   // timing experiment only (results are wrong): 8 warps, the last 15 packed covariance elements aliased
template <typename T> struct BlockOf { static constexpr int value = (sizeof(T) == 4) ? 384 : 256; };
#else
#ifndef QEKF_FP32_BLOCK
#define QEKF_FP32_BLOCK 384
#endif
template <typename T> struct BlockOf { static constexpr int value = (sizeof(T) == 4) ? QEKF_FP32_BLOCK : 224; };
#endif

template <typename T, bool BIAS, bool DIRECT, bool SYNTH, bool MR, bool PF, bool STATS>
cudaError_t launch_run(const RunArgs<T> &a, unsigned grid, size_t smem, cudaStream_t stream);

template <typename T, bool BIAS, bool PF>
cudaError_t launch_deliver(const DeviceState<T> &st, const Consts<T> &c, const double *pose8, int force_init,
                           int reinit_bias, int raise_ready, unsigned grid, size_t smem, cudaStream_t stream);

// the fused per-tick path of the N = 1 drop-in (tick_kernel); handles without per-filter overrides
template <typename T, bool BIAS, bool DIRECT, bool MR>
cudaError_t launch_tick(const RunArgs<T> &a, const double *pose8, int tag_mode, double *out, int n_out, cudaStream_t stream);

template <typename T, bool BIAS, bool PF>
cudaError_t launch_predict(const DeviceState<T> &st, const Consts<T> &c, const double *u, unsigned grid, size_t smem,
                           cudaStream_t stream);

template <typename T, bool BIAS, bool DIRECT, bool PF>
cudaError_t launch_correct(const DeviceState<T> &st, const Consts<T> &c, const double *tag, unsigned grid, size_t smem,
                           cudaStream_t stream);

template <typename T>
cudaError_t launch_reset(const DeviceState<T> &st, const Consts<T> &c, int nstates, int reset_nominal, cudaStream_t stream);

// history <- current head for every filter (checkpoint = x / P, no entries after it)
template <typename T> cudaError_t launch_rebase(const DeviceState<T> &st, int np, cudaStream_t stream);

template <typename T>
cudaError_t launch_dump(const RunArgs<T> &a, int64_t first, int64_t count, int64_t T_ticks, double *imu_out,
                        double *tag_out, uint8_t *valid_out, double *bias_out, cudaStream_t stream);

// column reordering of a [rows][ld] array of 4- / 8-byte words (W = uint32_t / uint64_t): filter order <-> slot order
template <typename W>
cudaError_t launch_permute_rows(W *dst, const W *src, const int32_t *perm, int64_t rows, int64_t ld, int64_t n, bool to_slots,
                                cudaStream_t stream);

// independent FMA chains, no memory traffic: `iters` x 16 FMAs per thread
template <typename T> cudaError_t launch_fma_peak(T *sink, int iters, unsigned grid, unsigned block, cudaStream_t stream);

// acc [STAT_REPL][n][STAT_DIM] -> out [n][STAT_DIM]
cudaError_t launch_stats_reduce(const double *acc, double *out, int64_t n, cudaStream_t stream);

template <typename K> inline cudaError_t prep_kernel(K kernel, size_t smem)
{
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}

}  // namespace qekf
