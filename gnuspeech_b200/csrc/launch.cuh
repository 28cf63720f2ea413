// launch.cuh -- per-precision launch wrappers.  Each kernels_*.cu translation unit instantiates these
// for one Real type (the FP64 conformance TU is compiled with -fmad=false, the FP32 TU with FMA
// contraction) and exports them with C linkage for trm_cuda.cu.
#pragma once

#include <stdlib.h>

#include "src_kernel.cuh"
#include "tube_wide.cuh"

namespace TRM_KERNEL_NS {
using namespace trm;

template <typename R, int SHAPE> constexpr int src_smem_bytes()
{
    using Cfg = SrcCfg<R, SHAPE>;
    return (Cfg::WINDOWS * 32 * Cfg::U * Cfg::XLD + Cfg::CBUFS * Cfg::NT_MAX * SRC_CLD + (Cfg::THREADS / 32) * 32 * Cfg::U * (SRC_CHUNK + 1)) *
           (int)sizeof(R);
}

template <typename R, int SHAPE> static int configure_src(KernelInfo *info)
{
    using Cfg = SrcCfg<R, SHAPE>;
    const int smem = src_smem_bytes<R, SHAPE>();
    cudaError_t e = cudaFuncSetAttribute(src_kernel<R, SHAPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    e = cudaFuncSetAttribute(src_kernel<R, SHAPE>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return (int)e;
    if (info) {
        KernelInfo::SrcShape &sh = info->src[SHAPE];
        sh.smem_bytes = smem; sh.threads = Cfg::THREADS; sh.tile = 32 * Cfg::U; sh.rows = Cfg::ROWS; sh.nt_max = Cfg::NT_MAX;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sh.ctas_per_sm, src_kernel<R, SHAPE>, Cfg::THREADS, smem);
        if (e != cudaSuccess) return (int)e;
        cudaFuncAttributes fa;
        if (cudaFuncGetAttributes(&fa, src_kernel<R, SHAPE>) == cudaSuccess) sh.regs = fa.numRegs;
    }
    return 0;
}

template <typename R> static int configure_kernels(KernelInfo *info)
{
    cudaError_t e;
    {
        int rc = configure_src<R, 0>(info);
        if (rc != 0) return rc;
        if constexpr (SrcShapes<R>::N == 2) {
            if ((rc = configure_src<R, 1>(info)) != 0) return rc;
        }
        if (info) info->n_src_shapes = SrcShapes<R>::N;
    }
    const int wide_smem = (int)sizeof(WideSmem<R>);
    for (auto k : {tube_wide_kernel<R, false>, tube_wide_kernel<R, true>}) {
        e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, wide_smem);
        if (e != cudaSuccess) return (int)e;
        e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return (int)e;
    }
    if (info) {
        info->wide_smem_bytes = wide_smem;
        info->wide_threads = Wide<R>::THREADS;
        info->wide_max_utt = 2 * Wide<R>::MAX_PAIRS;
        cudaFuncAttributes fa;
        if (cudaFuncGetAttributes(&fa, tube_wide_kernel<R, false>) == cudaSuccess) info->wide_regs = fa.numRegs;
        if (cudaFuncGetAttributes(&fa, pcm_kernel<R>) == cudaSuccess) info->pcm_regs = fa.numRegs;
    }
    return 0;
}

static int upload_constants(const double *fir, int taps, const unsigned long long *noise_pow)
{
    if (taps != FIR_TAPS) return -1;
    float firf[FIR_TAPS];
    for (int i = 0; i < FIR_TAPS; ++i) firf[i] = (float)fir[i];
    cudaError_t e = cudaMemcpyToSymbol(c_fir_d, fir, sizeof(double) * FIR_TAPS);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyToSymbol(c_fir_f, firf, sizeof(float) * FIR_TAPS);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyToSymbol(c_noise_pow, noise_pow, sizeof(unsigned long long) * (TRM_NOISE_JUMP + 1));
    return (int)e;
}

// waveguide: one CTA per group of <= 2*MAX_PAIRS utterances (tube_wide.cuh); per_utt: state stored per utterance (pools)
template <typename R> static int launch_tube_wide(const TubeArgs &a, int n_groups, cudaStream_t s, bool per_utt = false)
{
    if (a.n_utt <= 0 || n_groups <= 0) return 0;
    if ((a.n_utt + n_groups - 1) / n_groups > 2 * Wide<R>::MAX_PAIRS) return (int)cudaErrorInvalidConfiguration;
    WideArgs w{a, n_groups};
    if (per_utt) tube_wide_kernel<R, true><<<n_groups, Wide<R>::THREADS, sizeof(WideSmem<R>), s>>>(w);
    else tube_wide_kernel<R, false><<<n_groups, Wide<R>::THREADS, sizeof(WideSmem<R>), s>>>(w);
    return (int)cudaGetLastError();
}

template <typename R> static int launch_src(const SrcArgs &a, int grid, int shape, cudaStream_t s)
{
    const long long items = (a.item_end > 0 ? a.item_end : a.total_items) - a.item_begin;
    if (items <= 0) return 0;
    if ((long long)grid > items) grid = (int)items;
    if (shape == 0) {
        src_kernel<R, 0><<<grid, SrcCfg<R, 0>::THREADS, src_smem_bytes<R, 0>(), s>>>(a);
    } else if (shape == 1 && SrcShapes<R>::N == 2) {
        if constexpr (SrcShapes<R>::N == 2) src_kernel<R, 1><<<grid, SrcCfg<R, 1>::THREADS, src_smem_bytes<R, 1>(), s>>>(a);
    } else {
        return (int)cudaErrorInvalidValue;
    }
    return (int)cudaGetLastError();
}

template <typename R> static int launch_src_pool(const SrcPoolArgs &a, int grid, cudaStream_t s)
{
    if (a.total_items <= 0 || a.n <= 0) return 0;
    const long long need = (a.total_items + 7) / 8;                      // 8 warps per CTA, one work item per warp
    if ((long long)grid > need) grid = (int)need;
    src_pool_kernel<R><<<grid, 256, 0, s>>>(a);
    return (int)cudaGetLastError();
}

template <typename R> static int launch_pcm_pool(const PcmPoolArgs &a, int grid, cudaStream_t s)
{
    if (a.total_items <= 0 || a.n <= 0) return 0;
    const long long need = (a.total_items + 7) / 8;                      // 8 warps per CTA, one work item per warp
    if ((long long)grid > need) grid = (int)need;
    pcm_pool_kernel<R><<<grid, 256, 0, s>>>(a);
    return (int)cudaGetLastError();
}

template <typename R> static int launch_src_ctab(const void *tab, void *ctab, cudaStream_t s)
{
    const unsigned n = 65536u * SRC_CLD;
    src_ctab_kernel<R><<<(n + 255) / 256, 256, 0, s>>>(reinterpret_cast<const HD<R> *>(tab), reinterpret_cast<R *>(ctab));
    return (int)cudaGetLastError();
}

template <typename R> static int launch_pcm(const PcmArgs &a, long long max_n_out, cudaStream_t s)
{
    if (a.n_utt - a.u_begin <= 0 || max_n_out <= 0) return 0;
    const long long per_cta = (long long)PCM_THREADS * PCM_PER_THREAD;
    const long long bpu = (max_n_out + per_cta - 1) / per_cta;
    if (bpu > 0x7FFFFFFFll) return (int)cudaErrorInvalidConfiguration;
    dim3 grid((unsigned)bpu, (unsigned)(a.n_utt - a.u_begin < 65535 ? a.n_utt - a.u_begin : 65535));
    pcm_kernel<R><<<grid, PCM_THREADS, 0, s>>>(a);
    return (int)cudaGetLastError();
}

}  // namespace TRM_KERNEL_NS

#define TRM_DEFINE_LAUNCHERS(R, SUF)                                                                              \
    extern "C" int trm_k_configure_##SUF(trm::KernelInfo *info) { return TRM_KERNEL_NS::configure_kernels<R>(info); }      \
    extern "C" int trm_k_upload_##SUF(const double *fir, int taps, const unsigned long long *np)                 \
    {                                                                                                             \
        return TRM_KERNEL_NS::upload_constants(fir, taps, np);                                                              \
    }                                                                                                             \
    extern "C" int trm_k_tube_wide_##SUF(const trm::TubeArgs *a, int n_groups, cudaStream_t s)                    \
    {                                                                                                             \
        return TRM_KERNEL_NS::launch_tube_wide<R>(*a, n_groups, s);                                                         \
    }                                                                                                             \
    extern "C" int trm_k_tube_wide_pool_##SUF(const trm::TubeArgs *a, int n_groups, cudaStream_t s)               \
    {                                                                                                             \
        return TRM_KERNEL_NS::launch_tube_wide<R>(*a, n_groups, s, true);                                                   \
    }                                                                                                             \
    extern "C" int trm_k_src_##SUF(const trm::SrcArgs *a, int grid, int shape, cudaStream_t s)                    \
    {                                                                                                             \
        return TRM_KERNEL_NS::launch_src<R>(*a, grid, shape, s);                                                            \
    }                                                                                                             \
    extern "C" int trm_k_src_pool_##SUF(const trm::SrcPoolArgs *a, int grid, cudaStream_t s)                       \
    {                                                                                                             \
        return TRM_KERNEL_NS::launch_src_pool<R>(*a, grid, s);                                                              \
    }                                                                                                             \
    extern "C" int trm_k_pcm_pool_##SUF(const trm::PcmPoolArgs *a, int grid, cudaStream_t s)                       \
    {                                                                                                             \
        return TRM_KERNEL_NS::launch_pcm_pool<R>(*a, grid, s);                                                              \
    }                                                                                                             \
    extern "C" int trm_k_src_ctab_##SUF(const void *tab, void *ctab, cudaStream_t s)                              \
    {                                                                                                             \
        return TRM_KERNEL_NS::launch_src_ctab<R>(tab, ctab, s);                                                             \
    }                                                                                                             \
    extern "C" int trm_k_pcm_##SUF(const trm::PcmArgs *a, long long max_n_out, cudaStream_t s)                    \
    {                                                                                                             \
        return TRM_KERNEL_NS::launch_pcm<R>(*a, max_n_out, s);                                                              \
    }
