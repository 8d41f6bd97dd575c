// sp_inst.cuh — per-format instantiation of the render / pre-pass kernels.
// Each sp_inst_<fmt>.cu defines SP_INST_FMT and SP_INST_TAG and includes this file; it exports the format's launchers as one
// struct, sp_kernels_<tag>, which the engine binds through a weak symbol, so a build may carry any subset of specialised formats
// next to the runtime-switch variant (tag "rt").
#pragma once
#include "sp_kernels.cuh"
#include "sp_kernel_r64.cuh"
#include "sp_kernel_rc.cuh"
#include "sp_kernel_big.cuh"
#include "sp_kernel_w.cuh"

namespace sp {

// The launchers of one format's build.  A launcher given occ_out answers an occupancy probe (blocks per SM) and launches
// nothing; a kernel that is not built for the format answers 0.
struct Kernels {
    cudaError_t (*render)(int log2n, const Params *p, int grid, size_t smem, cudaStream_t st, int *occ_out);
    cudaError_t (*prepass)(int r, const Params *p, float2 *out, const float2 *tw_full, cudaStream_t st);
    cudaError_t (*r64)(int sub, const Params *p, int grid, cudaStream_t st, const float2 *tw14, const CUtensorMap *tm, int pdl, int *occ_out);
    cudaError_t (*rc)(int log2n, const Params *p, int grid, cudaStream_t st, const float2 *tw14, int *occ_out);
    cudaError_t (*w)(int log2n, const Params *p, int grid, cudaStream_t st, const float2 *twW, int *occ_out);
    cudaError_t (*big)(const Params *p, const BigArgs *g, int grid, cudaStream_t st, const float2 *tw14, int *occ_out);
};

// One launch of kernel K (or, with occ_out, its occupancy probe).  The dynamic shared-memory limit is set once per device:
// function attributes belong to the device's context, and a multi-device engine (sp_create with ndev > 1) launches the same
// kernel on several.  The flag is per kernel, so K is the kernel itself: instantiations of one kernel template may share a
// function type.  pdl: the launch may start before the kernel ahead of it in the stream has completed (programmatic
// dependent launch; the engine decides when that is safe).
template <auto K, typename... Args>
static cudaError_t launch_kernel(int grid, int threads, size_t smem, int smem_max, bool pdl, cudaStream_t st, int *occ_out,
                                 const Args &...args)
{
    static bool attr_done[64] = {};
    int d = 0;
    cudaGetDevice(&d);
    if (!attr_done[d & 63]) {
        cudaError_t e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
        if (e != cudaSuccess) return e;
        attr_done[d & 63] = true;
    }
    if (occ_out) return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ_out, K, threads, smem);
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = &attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, K, args...);
}

template <int LOG2N, int FMT>
static cudaError_t launch_one(const Params &p, int grid, size_t smem, cudaStream_t st, int *occ_out)
{
    return launch_kernel<render_kernel<LOG2N, FMT>>(grid, 256, smem, 200 * 1024, false, st, occ_out, p);
}

template <int FMT>
static cudaError_t launch_render(int log2n, const Params *p, int grid, size_t smem, cudaStream_t st, int *occ_out)
{
    switch (log2n) {
    case 1: return launch_one<1, FMT>(*p, grid, smem, st, occ_out);
    case 2: return launch_one<2, FMT>(*p, grid, smem, st, occ_out);
    case 3: return launch_one<3, FMT>(*p, grid, smem, st, occ_out);
    case 4: return launch_one<4, FMT>(*p, grid, smem, st, occ_out);
    case 5: return launch_one<5, FMT>(*p, grid, smem, st, occ_out);
    case 6: return launch_one<6, FMT>(*p, grid, smem, st, occ_out);
    case 7: return launch_one<7, FMT>(*p, grid, smem, st, occ_out);
    case 8: return launch_one<8, FMT>(*p, grid, smem, st, occ_out);
    case 9: return launch_one<9, FMT>(*p, grid, smem, st, occ_out);
    case 10: return launch_one<10, FMT>(*p, grid, smem, st, occ_out);
    case 11: return launch_one<11, FMT>(*p, grid, smem, st, occ_out);
    case 12: return launch_one<12, FMT>(*p, grid, smem, st, occ_out);
    default: return cudaErrorInvalidValue;
    }
}

template <int FMT>
static cudaError_t launch_prepass(int r, const Params *pp, float2 *out, const float2 *tw_full, cudaStream_t st)
{
    const Params &p = *pp;
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

// N = 4096 "64 x 64" path: one CTA of 4 x 64 threads per SM, 16 frames per tile (sp_kernel_r64.cuh)
template <int FMT, bool SUB, bool OPT>
static cudaError_t launch_r64_k(const Params &p, int grid, cudaStream_t st, const float2 *tw14, const CUtensorMap *tm, int pdl, int *occ_out)
{
    using B = R64Cfg<FMT, SUB>;
    return launch_kernel<render_r64_kernel<FMT, SUB, OPT>>(grid, B::THREADS, B::SMEM_BYTES, B::SMEM_BYTES, pdl, st, occ_out, p, tw14, *tm);
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
template <int FMT>
static cudaError_t launch_r64(int sub, const Params *p, int grid, cudaStream_t st, const float2 *tw14, const CUtensorMap *tm, int pdl, int *occ_out)
{
    if constexpr (FMT == CF32 || FMT == FMT_RUNTIME) {
        if (sub) return launch_r64_v<FMT, true>(*p, grid, st, tw14, tm, pdl, occ_out);
    } else if (sub) return cudaErrorInvalidValue;
    return launch_r64_v<FMT, false>(*p, grid, st, tw14, tm, pdl, occ_out);
}

// N = 2048 as 64 x 32 (sp_kernel_rc.cuh): same CTA shape as the 64 x 64 kernel.  N = 256 .. 1024 go to render_w_kernel.
template <int FMT>
static cudaError_t launch_rc(int log2n, const Params *p, int grid, cudaStream_t st, const float2 *tw14, int *occ_out)
{
    using B = RcCfg<FMT>;
    if (log2n != 11) return cudaErrorInvalidValue;
    if constexpr (!B::OK) {
        if (occ_out) *occ_out = 0;
        return occ_out ? cudaSuccess : cudaErrorInvalidValue;
    } else {
        return launch_kernel<render_rc_kernel<FMT>>(grid, B::THREADS, B::SMEM_BYTES, B::SMEM_BYTES, false, st, occ_out, *p, tw14);
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
        if (p.channel_mode)
            return launch_kernel<render_w_kernel<LOG2P, LOG2T, FMT, true>>(grid, B::THREADS, B::SMEM_BYTES, B::SMEM_BYTES, false, st, occ_out, p, twW);
        return launch_kernel<render_w_kernel<LOG2P, LOG2T, FMT, false>>(grid, B::THREADS, B::SMEM_BYTES, B::SMEM_BYTES, false, st, occ_out, p, twW);
    }
}
template <int FMT>
static cudaError_t launch_w(int log2n, const Params *p, int grid, cudaStream_t st, const float2 *twW, int *occ_out)
{
    switch (log2n) {
    case 6: return launch_w_v<3, 3, FMT>(*p, grid, st, twW, occ_out);
    case 7: return launch_w_v<4, 3, FMT>(*p, grid, st, twW, occ_out);
    case 8: return launch_w_v<4, 4, FMT>(*p, grid, st, twW, occ_out);
    case 9: return launch_w_v<5, 4, FMT>(*p, grid, st, twW, occ_out);
    case 10: return launch_w_v<5, 5, FMT>(*p, grid, st, twW, occ_out);
    default: return cudaErrorInvalidValue;
    }
}

// n = R * 4096 in one persistent launch (sp_kernel_big.cuh)
template <int FMT>
static cudaError_t launch_big(const Params *p, const BigArgs *g, int grid, cudaStream_t st, const float2 *tw14, int *occ_out)
{
    return launch_kernel<render_big_kernel<FMT>>(grid, BigCfg::THREADS, BigCfg::SMEM_BYTES, BigCfg::SMEM_BYTES, false, st, occ_out, *p, *g, tw14);
}

} // namespace sp

#ifdef SP_INST_FMT
#define SP_CAT2(a, b) a##b
#define SP_CAT(a, b) SP_CAT2(a, b)
extern "C" const sp::Kernels SP_CAT(sp_kernels_, SP_INST_TAG) = {
    sp::launch_render<SP_INST_FMT>, sp::launch_prepass<SP_INST_FMT>, sp::launch_r64<SP_INST_FMT>,
    sp::launch_rc<SP_INST_FMT>,     sp::launch_w<SP_INST_FMT>,       sp::launch_big<SP_INST_FMT> };
#endif
