// sp_inst.cuh — per-format instantiation of the render / pre-pass kernels.
// Each sp_inst_<fmt>.cu defines SP_INST_FMT and SP_INST_TAG and includes this file; the engine
// binds the resulting entry points through weak symbols, so a build may carry any subset of
// specialised formats next to the runtime-switch variant (tag "rt").
#pragma once
#include "sp_kernels.cuh"
#include "sp_kernel_r64.cuh"
#include "sp_kernel_rc.cuh"
#include "sp_kernel_big.cuh"
#include "sp_kernel_w.cuh"

namespace sp {

// cudaFuncSetAttribute is per device: a multi-device engine (sp_create with ndev > 1) launches the same kernel on several
static inline bool &attr_flag(bool (&flags)[64])
{
    int d = 0;
    cudaGetDevice(&d);
    return flags[d & 63];
}

template <int LOG2N, int FMT>
static cudaError_t launch_one(const Params &p, int grid, size_t smem, cudaStream_t st, int *occ_out)
{
    auto kfn = render_kernel<LOG2N, FMT>;
    static bool attr_flags[64] = {};         // per device: function attributes belong to the device's context
    bool &attr_done = attr_flag(attr_flags);
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_done = true;
    }
    if (occ_out) {
        int nb = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kfn, 256, smem);
        *occ_out = nb;
        return e;
    }
    kfn<<<grid, 256, smem, st>>>(p);
    return cudaGetLastError();
}

template <int FMT>
static cudaError_t launch_render(int log2n, const Params &p, int grid, size_t smem, cudaStream_t st, int *occ_out)
{
    switch (log2n) {
    case 1: return launch_one<1, FMT>(p, grid, smem, st, occ_out);
    case 2: return launch_one<2, FMT>(p, grid, smem, st, occ_out);
    case 3: return launch_one<3, FMT>(p, grid, smem, st, occ_out);
    case 4: return launch_one<4, FMT>(p, grid, smem, st, occ_out);
    case 5: return launch_one<5, FMT>(p, grid, smem, st, occ_out);
    case 6: return launch_one<6, FMT>(p, grid, smem, st, occ_out);
    case 7: return launch_one<7, FMT>(p, grid, smem, st, occ_out);
    case 8: return launch_one<8, FMT>(p, grid, smem, st, occ_out);
    case 9: return launch_one<9, FMT>(p, grid, smem, st, occ_out);
    case 10: return launch_one<10, FMT>(p, grid, smem, st, occ_out);
    case 11: return launch_one<11, FMT>(p, grid, smem, st, occ_out);
    case 12: return launch_one<12, FMT>(p, grid, smem, st, occ_out);
    default: return cudaErrorInvalidValue;
    }
}

template <int FMT>
static cudaError_t launch_prepass(int r, const Params &p, float2 *out, const float2 *tw_full, cudaStream_t st)
{
    const long long threads = p.chunk_frames * 4096;
    const int grid = (int)((threads + 255) / 256);
    switch (r) {
    case 2: prepass_kernel<2, FMT><<<grid, 256, 0, st>>>(p, out, tw_full); break;
    case 4: prepass_kernel<4, FMT><<<grid, 256, 0, st>>>(p, out, tw_full); break;
    case 8: prepass_kernel<8, FMT><<<grid, 256, 0, st>>>(p, out, tw_full); break;
    case 16: prepass_kernel<16, FMT><<<grid, 256, 0, st>>>(p, out, tw_full); break;
    case 32: prepass_kernel<32, FMT><<<grid, 256, 0, st>>>(p, out, tw_full); break;
    case 64: prepass_kernel<64, FMT><<<grid, 256, 0, st>>>(p, out, tw_full); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// N = 4096 "64 x 64" path: one CTA of 4 x 64 threads per SM, 16 frames per tile (sp_kernel_r64.cuh).  pdl: the launch may start
// before the kernel ahead of it in the stream has completed (programmatic dependent launch; the engine decides when that is safe).
template <int FMT, bool SUB, bool OPT>
static cudaError_t launch_r64_k(const Params &p, int grid, cudaStream_t st, const float2 *tw14, const CUtensorMap *tm, int pdl, int *occ_out)
{
    using B = R64Cfg<FMT, SUB>;
    auto kfn = render_r64_kernel<FMT, SUB, OPT>;
    static bool attr_flags[64] = {};
    bool &attr_done = attr_flag(attr_flags);
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        attr_done = true;
    }
    if (occ_out) {
        int nb = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kfn, B::THREADS, B::SMEM_BYTES);
        *occ_out = nb;
        return e;
    }
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(B::THREADS);
    cfg.dynamicSmemBytes = B::SMEM_BYTES;
    cfg.stream = st;
    cfg.attrs = &attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kfn, p, tw14, *tm);
}
template <int FMT, bool SUB>
static cudaError_t launch_r64_v(const Params &p, int grid, cudaStream_t st, const float2 *tw14, const CUtensorMap *tm, int pdl, int *occ_out)
{
    using B = R64Cfg<FMT, SUB>;
    if constexpr (!B::OK) {
        if (occ_out) *occ_out = 0;
        return occ_out ? cudaSuccess : cudaErrorInvalidValue;
    } else if constexpr (SUB) {
        return launch_r64_k<FMT, true, false>(p, grid, st, tw14, tm, pdl, occ_out);
    } else {
        // messages that ask for the waterfall layout or the split-real post-process take the kernel compiled with them
        if (p.waterfall || p.channel_mode) return launch_r64_k<FMT, false, true>(p, grid, st, tw14, tm, pdl, occ_out);
        return launch_r64_k<FMT, false, false>(p, grid, st, tw14, tm, pdl, occ_out);
    }
}

// N = 512 / 1024 / 2048 as 64 x C (sp_kernel_rc.cuh): same CTA shape as the 64 x 64 kernel.
template <int LOG2C, int FMT>
static cudaError_t launch_rc_v(const Params &p, int grid, cudaStream_t st, const float2 *tw14, int *occ_out)
{
    using B = RcCfg<LOG2C, FMT>;
    if constexpr (!B::OK) {
        if (occ_out) *occ_out = 0;
        return occ_out ? cudaSuccess : cudaErrorInvalidValue;
    } else {
        auto kfn = render_rc_kernel<LOG2C, FMT>;
        static bool attr_flags[64] = {};
        bool &attr_done = attr_flag(attr_flags);
        if (!attr_done) {
            cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B::SMEM_BYTES);
            if (e != cudaSuccess) return e;
            attr_done = true;
        }
        if (occ_out) {
            int nb = 0;
            cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kfn, B::THREADS, B::SMEM_BYTES);
            *occ_out = nb;
            return e;
        }
        kfn<<<grid, B::THREADS, B::SMEM_BYTES, st>>>(p, tw14);
        return cudaGetLastError();
    }
}

// N = 64 .. 1024 as P x T, one warp per FW frames (sp_kernel_w.cuh)
template <int LOG2P, int LOG2T, int FMT>
static cudaError_t launch_w_v(const Params &p, int grid, cudaStream_t st, const float2 *twW, int *occ_out)
{
    using B = WCfg<LOG2P, LOG2T, FMT>;
    if constexpr (!B::OK) {
        if (occ_out) *occ_out = 0;
        return occ_out ? cudaSuccess : cudaErrorInvalidValue;
    } else {
        // channelMode messages take the instantiation that carries the split-real post-process
        auto kfn = p.channel_mode ? render_w_kernel<LOG2P, LOG2T, FMT, true> : render_w_kernel<LOG2P, LOG2T, FMT, false>;
        static bool attr_flags[2][64] = {};
        bool &attr_done = attr_flag(attr_flags[p.channel_mode ? 1 : 0]);
        if (!attr_done) {
            cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B::SMEM_BYTES);
            if (e != cudaSuccess) return e;
            attr_done = true;
        }
        if (occ_out) {
            int nb = 0;
            cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kfn, B::THREADS, B::SMEM_BYTES);
            *occ_out = nb;
            return e;
        }
        kfn<<<grid, B::THREADS, B::SMEM_BYTES, st>>>(p, twW);
        return cudaGetLastError();
    }
}

// n = R * 4096 in one persistent launch (sp_kernel_big.cuh)
template <int FMT>
static cudaError_t launch_big_v(const Params &p, const BigArgs &g, int grid, cudaStream_t st, const float2 *tw14, int *occ_out)
{
    auto kfn = render_big_kernel<FMT>;
    static bool attr_flags[64] = {};
    bool &attr_done = attr_flag(attr_flags);
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BigCfg::SMEM_BYTES);
        if (e != cudaSuccess) return e;
        attr_done = true;
    }
    if (occ_out) {
        int nb = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kfn, BigCfg::THREADS, BigCfg::SMEM_BYTES);
        *occ_out = nb;
        return e;
    }
    kfn<<<grid, BigCfg::THREADS, BigCfg::SMEM_BYTES, st>>>(p, g, tw14);
    return cudaGetLastError();
}

} // namespace sp

#define SP_CAT2(a, b) a##b
#define SP_CAT(a, b) SP_CAT2(a, b)

#ifdef SP_INST_FMT
extern "C" cudaError_t SP_CAT(sp_rl_, SP_INST_TAG)(int log2n, const sp::Params *p, int grid, size_t smem,
                                                    cudaStream_t st, int *occ_out)
{
    return sp::launch_render<SP_INST_FMT>(log2n, *p, grid, smem, st, occ_out);
}
extern "C" cudaError_t SP_CAT(sp_r64_, SP_INST_TAG)(int sub, const sp::Params *p, int grid, cudaStream_t st, const float2 *tw14, const CUtensorMap *tm,
                                                     int pdl, int *occ_out)
{
    if constexpr (SP_INST_FMT == sp::CF32 || SP_INST_FMT == sp::FMT_RUNTIME) {
        if (sub) return sp::launch_r64_v<SP_INST_FMT, true>(*p, grid, st, tw14, tm, pdl, occ_out);
    } else if (sub) return cudaErrorInvalidValue;
    return sp::launch_r64_v<SP_INST_FMT, false>(*p, grid, st, tw14, tm, pdl, occ_out);
}
extern "C" cudaError_t SP_CAT(sp_rc_, SP_INST_TAG)(int log2n, const sp::Params *p, int grid, cudaStream_t st, const float2 *tw14, int *occ_out)
{
    // N = 2048 only: render_w_kernel took over N = 256 .. 1024 in round 2 (both layouts); the template still covers C = 4 .. 32
    switch (log2n) {
    case 11: return sp::launch_rc_v<5, SP_INST_FMT>(*p, grid, st, tw14, occ_out);
    default: return cudaErrorInvalidValue;
    }
}
extern "C" cudaError_t SP_CAT(sp_w_, SP_INST_TAG)(int log2n, const sp::Params *p, int grid, cudaStream_t st, const float2 *twW, int *occ_out)
{
    switch (log2n) {
    case 6: return sp::launch_w_v<3, 3, SP_INST_FMT>(*p, grid, st, twW, occ_out);
    case 7: return sp::launch_w_v<4, 3, SP_INST_FMT>(*p, grid, st, twW, occ_out);
    case 8: return sp::launch_w_v<4, 4, SP_INST_FMT>(*p, grid, st, twW, occ_out);
    case 9: return sp::launch_w_v<5, 4, SP_INST_FMT>(*p, grid, st, twW, occ_out);
    case 10: return sp::launch_w_v<5, 5, SP_INST_FMT>(*p, grid, st, twW, occ_out);
    default: return cudaErrorInvalidValue;
    }
}
extern "C" cudaError_t SP_CAT(sp_big_, SP_INST_TAG)(const sp::Params *p, const sp::BigArgs *g, int grid, cudaStream_t st, const float2 *tw14, int *occ_out)
{
    return sp::launch_big_v<SP_INST_FMT>(*p, *g, grid, st, tw14, occ_out);
}
extern "C" cudaError_t SP_CAT(sp_pl_, SP_INST_TAG)(int r, const sp::Params *p, float2 *out, const float2 *tw_full,
                                                    cudaStream_t st)
{
    return sp::launch_prepass<SP_INST_FMT>(r, *p, out, tw_full, st);
}
#endif
