// sp_fused.cuh — the blocks that every fused render kernel (render_r64_kernel, render_rc_kernel, render_w_kernel,
// render_big_kernel) runs the same way: the CTA prologue (reversed colour LUT, cleared joint histogram),
// the per-bin epilogue of the FFT warps (|X|^2 -> min / max, joint-histogram atomic, colour byte), the fix-up of frames
// that hold zero / +inf / NaN magnitudes, the store warps' LUT look-ups and dB conversion, the pass-A twiddles of the
// 64-point kernels and the joint-histogram flush.  The kernels keep what differs between them: tile scheduling, staging
// layouts, the store warps' iteration orders, the FFT passes and the shared-memory carve-ups.
#pragma once
#include "sp_prims.cuh"

namespace sp {

// RGBA of byte j of a staged word: table base on a 1 KB boundary of the shared window
__device__ __forceinline__ unsigned lut_at(unsigned lut_base, unsigned word, int j)
{
    const unsigned a = ((j == 0 ? word << 2 : word >> (8 * j - 2)) & 0x3fcu) | lut_base;
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// byte j of 8 staged words (8 consecutive frames of one word column) as 8 RGBA pixels of one image row
__device__ __forceinline__ void lut_row8(unsigned lut_base, const unsigned (&w)[8], int j, uint4 &a, uint4 &b)
{
    a.x = lut_at(lut_base, w[0], j); a.y = lut_at(lut_base, w[1], j); a.z = lut_at(lut_base, w[2], j); a.w = lut_at(lut_base, w[3], j);
    b.x = lut_at(lut_base, w[4], j); b.y = lut_at(lut_base, w[5], j); b.z = lut_at(lut_base, w[6], j); b.w = lut_at(lut_base, w[7], j);
}

// one row segment of 8 pixels: a 256-bit store when every image row is 32-byte aligned (width % 8 == 0), else 8 words
__device__ __forceinline__ void store_row8(uint32_t *rowp, uint4 a, uint4 b, bool aligned)
{
    if (aligned) st_global_256(rowp, a, b);
    else {
        rowp[0] = a.x; rowp[1] = a.y; rowp[2] = a.z; rowp[3] = a.w;
        rowp[4] = b.x; rowp[5] = b.y; rowp[6] = b.z; rowp[7] = b.w;
    }
}

// the 64 threads of frame stream `stream` (named barrier stream + 1)
__device__ __forceinline__ void stream_barrier(int stream)
{
    asm volatile("bar.sync %0, 64;" ::"r"(stream + 1) : "memory");
}

// CTA prologue: clear the joint histogram, fill the reversed RGBA LUT (indexed by the staged byte: cmax - g, or g when
// range < 0; s_lut on the 1 KB boundary lut_at expects)
__device__ __forceinline__ JhConst fused_prologue(const Params &p, unsigned *s_jh, unsigned *s_lut, int tid, int nthreads)
{
    for (int i = tid; i < JH_SIZE; i += nthreads) s_jh[i] = 0;
    const int cmax = p.cmap_len - 1;
    const JhConst jc = jh_const(p);
    for (int i = tid; i < 256; i += nthreads) s_lut[i] = i <= cmax ? p.lut[jc.rev ? cmax - i : i] : 0u;
    return jc;
}

// min / max of |X|^2 over a thread's bins.  Float input (|X|^2 may be +inf / NaN): unsigned order on the bit patterns, where
// a NaN wins the max (and is sorted out by fixup_nonfinite), never the min.  Integer input: |X|^2 is finite and >= 0, its
// bit patterns order like the values, and a 3-input FMNMX3 takes two bins at a time.
template <bool FLOAT_IN> struct BinMinMax {
    float amin = __builtin_huge_valf(), amax = 0.0f, prev = 0.0f;
    unsigned umin = 0x7f800000u, umax = 0u;
    __device__ __forceinline__ unsigned lo() const { return FLOAT_IN ? umin : __float_as_uint(amin); }
    __device__ __forceinline__ unsigned hi() const { return FLOAT_IN ? umax : __float_as_uint(amax); }
};

// Per-bin epilogue (lib/worker.js:85-122) of the four bins q[0..3]: min / max, one joint-histogram atomic per bin (at
// jbase + 4 * (2^23 + joint index) when `live`, else at the unused counter `dump`), and the four colour bytes as one word.
template <bool FLOAT_IN>
__device__ __forceinline__ unsigned epilogue4(const cf *q, BinMinMax<FLOAT_IN> &mm, const JhConst &jc, unsigned jbase, bool live, unsigned dump)
{
    unsigned yb[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const float2 vi = cun(q[j]);
        const float abs2 = fmaf(vi.x, vi.x, vi.y * vi.y);
        if constexpr (FLOAT_IN) {
            mm.umin = min(mm.umin, __float_as_uint(abs2));
            mm.umax = max(mm.umax, __float_as_uint(abs2));
        } else if (j & 1) {
            mm.amin = fmin3(mm.amin, mm.prev, abs2);
            mm.amax = fmax3(mm.amax, mm.prev, abs2);
        } else mm.prev = abs2;
        const float l2 = fast_log2(abs2);
        float Y;
        const float S = jh_eval(l2, jc, Y);                     // 2^23 + joint index, 2^23 + (cmax - colour index)
        red_shared_inc_addr(live ? jbase + (__float_as_uint(S) << 2) : dump);
        yb[j] = __float_as_uint(Y);
    }
    return __byte_perm(__byte_perm(yb[0], yb[1], 0x0040), __byte_perm(yb[2], yb[3], 0x0040), 0x5410);
}

// Rare (called warp-uniformly, when umn / umx show |X|^2 == 0 (flushed: d0 = -inf), +inf or NaN in a frame of the warp):
// count those bins for the bin-0 fix-ups of finalize_kernel (lib/worker.js:105-106: ~~(+-Infinity) == ~~NaN == 0), move the
// NaN bins out of the joint index sat(NaN) = 0 yields, and redo umn / umx the way the reference's `<` / `>` see them (NaN
// never wins).  gmin / gmax reduce over the lanes of one frame; bins of lanes with count == false are not counted, and
// `leader` is the one lane of the warp that updates the histogram, which it skips when !live (a warp that holds one frame
// only may pass its frame's validity either way: render_r64_kernel compiles best with `live`).
template <int NP, typename GMin, typename GMax>
__device__ __forceinline__ void fixup_nonfinite(const cf (&v)[NP], bool count, bool leader, bool live, unsigned *s_jh, const JhConst &jc,
                                                GMin gmin, GMax gmax, unsigned &umn, unsigned &umx)
{
    unsigned nzero = 0, nbad = 0, nnan = 0;
    float mn = __int_as_float(0x7f800000), mx = 0.0f;
#pragma unroll
    for (int i = 0; i < NP; i++) {
        const float2 vi = cun(v[i]);
        const float abs2 = fmaf(vi.x, vi.x, vi.y * vi.y);
        nzero += abs2 < 1.17549435e-38f ? 1u : 0u;
        nbad += !(abs2 <= 3.402823466e38f) ? 1u : 0u;
        nnan += abs2 != abs2 ? 1u : 0u;
        mn = fminf(mn, abs2 < 1.17549435e-38f ? 0.0f : abs2);
        mx = fmaxf(mx, abs2);
    }
    if (!count) nzero = nbad = nnan = 0;
    nzero = __reduce_add_sync(0xffffffffu, nzero);
    nbad = __reduce_add_sync(0xffffffffu, nbad);
    nnan = __reduce_add_sync(0xffffffffu, nnan);
    umn = gmin(__float_as_uint(mn));
    umx = gmax(__float_as_uint(mx));
    if (leader && live) {
        if (nzero) atomicAdd(&s_jh[JH_ZERO], nzero);
        if (nbad) atomicAdd(&s_jh[JH_BAD], nbad);
        if (nnan) {
            float Yn;
            const float Sn = jh_eval(__int_as_float(0x7fffffff), jc, Yn);
            atomicSub(&s_jh[__float_as_uint(Sn) - JH_MAGIC_BITS], nnan);
            atomicAdd(&s_jh[JH_NAN], nnan);
        }
    }
}

// full-warp reducers for fixup_nonfinite (a frame spans whole warps)
struct WarpMin { __device__ __forceinline__ unsigned operator()(unsigned x) const { return __reduce_min_sync(0xffffffffu, x); } };
struct WarpMax { __device__ __forceinline__ unsigned operator()(unsigned x) const { return __reduce_max_sync(0xffffffffu, x); } };

// a frame's min / max bit patterns of |X|^2 as dB (lib/worker.js:82-83, 102-103): .x = min, .y = max
__device__ __forceinline__ float2 frame_db(unsigned umn, unsigned umx, const Params &p)
{
    return make_float2(fminf(0.0f, fmaf(fast_log2(__uint_as_float(umn)), p.c1, p.c0)),
                       fmaxf(-200.0f, fmaf(fast_log2(__uint_as_float(umx)), p.c1, p.c0)));
}

// End of pass A of the 64-point kernels: v[k] *= W^{t*k} (tw14 row of thread t: W^{t*k}, k = 1..7, 8, 16, .., 56; the
// others are formed as W^{t*8i} W^{t*j}), each product followed by its exchange store to dst(k), so that the stores ride
// between the FFMA2.  The upper twiddles are read after the first eight stores (render_rc_kernel reads all of them up front
// and keeps its own copy of this block: the two orders compile differently).
template <typename Dst>
__device__ __forceinline__ void twiddle_store64(cf (&v)[64], const float4 *twp, Dst dst)
{
    float2 w[8];                                                // w[j] = W^{t*j}, j = 1..7
    const float4 a = twp[0], b = twp[1], c = twp[2], d = twp[3];
    w[1] = make_float2(a.x, a.y); w[2] = make_float2(a.z, a.w); w[3] = make_float2(b.x, b.y); w[4] = make_float2(b.z, b.w);
    w[5] = make_float2(c.x, c.y); w[6] = make_float2(c.z, c.w); w[7] = make_float2(d.x, d.y);
#pragma unroll
    for (int j = 1; j < 8; j++) v[j] = cmul(v[j], w[j]);
#pragma unroll
    for (int k = 0; k < 8; k++) cst(dst(k), v[k]);
    float2 hi[8];                                               // hi[i] = W^{t*8i}, i = 1..7
    hi[1] = make_float2(d.z, d.w);
    const float4 e = twp[4], f = twp[5], g = twp[6];
    hi[2] = make_float2(e.x, e.y); hi[3] = make_float2(e.z, e.w); hi[4] = make_float2(f.x, f.y);
    hi[5] = make_float2(f.z, f.w); hi[6] = make_float2(g.x, g.y); hi[7] = make_float2(g.z, g.w);
#pragma unroll
    for (int i = 1; i < 8; i++) {
        v[8 * i] = cmul(v[8 * i], hi[i]);
#pragma unroll
        for (int j = 1; j < 8; j++) v[8 * i + j] = cmul(v[8 * i + j], cun(cmul(cpk(hi[i]), w[j])));
#pragma unroll
        for (int k = 8 * i; k < 8 * i + 8; k++) cst(dst(k), v[k]);
    }
}

// add the CTA's joint histogram to the render's (after a CTA barrier)
__device__ __forceinline__ void flush_joint_hist(const Params &p, const unsigned *s_jh, int tid, int nthreads)
{
    for (int i = tid; i < JH_SIZE; i += nthreads)
        if (s_jh[i]) atomicAdd(&p.j_hist[i], (unsigned long long)s_jh[i]);
}

} // namespace sp
